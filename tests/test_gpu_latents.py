"""GPU tests of the device latent stream (csrc/latent.cuh, include/pbg.h: pbg_draw_latents / pbg_set_latent_stream):
draws equal torch.randn on a CUDA generator bit for bit, and every generator entry point given z = None equals the same
call given that draw."""
import json

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

SEED = 20261020


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.fail("gpu-marked tests need a CUDA device (there is no CPU fallback to test)")
    assert torch.cuda.get_device_capability(0)[0] == 10, "kernels are sm_100a only"
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def cuda_models(dev, synth):
    import modular_prot_b_gan as m
    G, D = synth.make_models(m.ModularGenerator, m.ModularDiscriminator)
    return G.to(dev).eval(), D.to(dev).eval()


@pytest.fixture(scope="module")
def dev_tables(tables, dev):
    node_emb, rel_w = tables
    return node_emb.to(dev), rel_w.to(dev)


def twin(dev, seed=SEED, offset=0):
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    g.set_offset(offset)
    return g


def assert_bits_equal(got, want, what):
    if torch.equal(got, want):
        return
    gi, wi = got.reshape(-1).view(torch.int32), want.reshape(-1).view(torch.int32)
    i = int((gi != wi).nonzero()[0, 0])
    raise AssertionError(f"{what}: {int((gi != wi).sum())} elements differ; first at flat index {i}: "
                         f"got {got.reshape(-1)[i].item()!r} (0x{gi[i].item() & 0xffffffff:08x}), "
                         f"torch {want.reshape(-1)[i].item()!r} (0x{wi[i].item() & 0xffffffff:08x})")


# ----------------------------------------------------------------------------- the draw itself
ROWS = [1, 3, 16, 255, 4096, 4097, 18944, 18945, 32768, 65537, 150000]   # 18944 / 18945 cross a round at Z = 64
# A ctx's noise_dim is a multiple of 8 (pbg_create); the draw depends on rows and Z only through numel = rows * Z.
WIDTHS = [8, 24, 64, 256]
POSITIONS = [(SEED, 0), (7, 4 * 1000003), (2 ** 40 + 3, 2 ** 33)]


@pytest.mark.parametrize("Z", WIDTHS)
def test_draw_equals_torch_randn(dev, Z):
    from pbg.engine import Engine
    eng = Engine(8, Z, 8, 16, dev)
    for rows in ROWS:
        for seed, off in POSITIONS:
            g = twin(dev, seed, off)
            want = torch.randn((rows, Z), device=dev, generator=g)
            got, after = eng.draw_latents(rows, seed, off)
            assert_bits_equal(got, want, f"rows={rows} Z={Z} seed={seed} offset={off}")
            assert after == g.get_offset(), (rows, Z, seed, off)


@pytest.mark.parametrize("rows", [4097, 65537, 150000])
def test_row_ranges_concatenate_to_the_whole_draw(dev, rows):
    from pbg.engine import Engine
    eng = Engine(8, 64, 8, 16, dev)
    whole, after = eng.draw_latents(rows, SEED, 8)
    cuts = [0, 1, rows // 3, rows // 3 + 255, rows - 1, rows]
    parts = []
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        z, a = eng.draw_latents(hi - lo, SEED, 8, row_begin=lo, total_rows=rows)
        assert a == after
        parts.append(z)
    assert_bits_equal(torch.cat(parts), whole, f"row ranges of {rows}")
    with pytest.raises(Exception):
        eng.draw_latents(2, SEED, 8, row_begin=rows - 1, total_rows=rows)    # beyond the draw
    with pytest.raises(Exception):
        eng.draw_latents(4, SEED, 2)                                         # torch's offsets are multiples of 4


# ----------------------------------------------------------------------------- the ctx's stream in the passes
def _pass(eng, dev_tables, trip, z, precision="bf16", **kw):
    kw = kw or dict(want_gen_out=True, want_gen_scores=True, want_disc=True)
    return eng.score_triplets(*dev_tables, trip, z, precision=precision, **kw)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_score_triplets_without_z_draws_what_torch_draws(cuda_models, dev_tables, synth, dev, precision):
    import modular_prot_b_gan as m
    eng = m.make_fused_engine(*cuda_models)
    with pytest.raises(ValueError):
        _pass(eng, dev_tables, synth.make_triplets(4).to(dev), None, precision)   # stream off: refused as before
    eng.set_latent_stream(True, SEED, 0)
    g = twin(dev)
    for i, B in enumerate([5, 4096, 300, 70000, 1, 33]):
        trip = synth.make_triplets(B, seed=900 + i).to(dev)
        if i == 2:   # discriminator-only calls draw nothing
            _pass(eng, dev_tables, trip, None, precision, want_disc=True)
            assert eng.latent_stream() == (SEED, g.get_offset())
        got = {k: v.clone() for k, v in _pass(eng, dev_tables, trip, None, precision).items()}
        z = torch.randn((B, eng.Z), device=dev, generator=g)
        want = _pass(eng, dev_tables, trip, z, precision)                 # caller latents: the stream stays put
        for k in want:
            assert_bits_equal(got[k], want[k], f"B={B} {precision} {k}")
        assert eng.latent_stream() == (SEED, g.get_offset()), B
    eng.check_indices()
    # generator-only entry points draw the same way
    h, r = dev_tables[0][:100], dev_tables[1][torch.arange(100, device=dev) % 64]
    got = eng.generator_forward(h, r, precision=precision)
    assert torch.equal(got, eng.generator_forward(h, r, torch.randn((100, eng.Z), device=dev, generator=g), precision=precision))
    heads, rels = torch.arange(50, device=dev), torch.arange(50, device=dev) % 64
    got = eng.generator_forward_gather(*dev_tables, heads, rels, precision=precision)
    want = eng.generator_forward_gather(*dev_tables, heads, rels, torch.randn((50, eng.Z), device=dev, generator=g),
                                        precision=precision)
    assert torch.equal(got, want)
    assert eng.latent_stream() == (SEED, g.get_offset())


def test_staged_lanes_draw_in_staging_order(cuda_models, dev_tables, synth, dev):
    import modular_prot_b_gan as m
    sizes = [1000, 4096, 31, 257, 5000]
    eng = m.make_fused_engine(*cuda_models, ctas=48)
    trips = [synth.make_triplets(B, seed=700 + i).to(dev) for i, B in enumerate(sizes)]
    g = twin(dev)
    zs = [torch.randn((B, eng.Z), device=dev, generator=g) for B in sizes]   # staging order
    kw = dict(want_gen_out=True, want_gen_scores=True, want_disc=True, out_dtype=torch.bfloat16)
    ref = [{k: v.clone() for k, v in _pass(eng, dev_tables, t, z, out_dtype=torch.bfloat16,
                                           want_gen_out=True, want_gen_scores=True, want_disc=True).items()}
           for t, z in zip(trips, zs)]
    eng.reserve(max(sizes), "bf16", 2)
    # stage, then score, one request at a time
    eng.set_latent_stream(True, SEED, 0)
    for j, t in enumerate(trips):
        eng.stage_triplets(j & 1, *dev_tables, t)
        res = eng.score_staged(j & 1, **kw)
        for k in ref[j]:
            assert_bits_equal(res[k], ref[j][k], f"staged request {j}: {k}")
    assert eng.latent_stream()[1] == g.get_offset()
    # the pass that stages the next request draws that request's latents
    eng.set_latent_stream(True, SEED, 0)
    eng.stage_triplets(0, *dev_tables, trips[0])
    got = []
    for j in range(len(trips)):
        nxt = (*dev_tables, trips[j + 1], None) if j + 1 < len(trips) else None
        got.append(eng.score_staged(j & 1, stage_next=nxt, **kw))
    torch.cuda.synchronize()
    eng.check_indices()
    for j in range(len(trips)):
        for k in ref[j]:
            assert_bits_equal(got[j][k], ref[j][k], f"stage-next request {j}: {k}")
    assert eng.latent_stream()[1] == g.get_offset()


def test_captured_lane_draws_fresh_latents_on_every_replay(cuda_models, dev_tables, synth, dev):
    import modular_prot_b_gan as m
    sizes = [4096, 700, 2048]
    eng = m.make_fused_engine(*cuda_models, ctas=48)
    eng.reserve(max(sizes), "bf16", 0)
    trips = [synth.make_triplets(B, seed=40 + i).to(dev) for i, B in enumerate(sizes)]
    kw = dict(want_gen_out=True, want_gen_scores=True, want_disc=True)
    outs = [{"gen_out": torch.zeros(B, eng.E, device=dev), "gen_scores": torch.zeros(B, device=dev),
             "logits": torch.zeros(B, device=dev), "probs": torch.zeros(B, device=dev)} for B in sizes]
    eng.set_latent_stream(True, SEED, 0)
    cs = torch.cuda.Stream(dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(cs):
        with torch.cuda.graph(graph, stream=cs):
            for t, o in zip(trips, outs):
                eng.score_triplets(*dev_tables, t, None, out=o, **kw)
    assert eng.latent_stream() == (SEED, 0)            # capturing draws nothing
    g = twin(dev)
    for rep in range(2):
        with torch.cuda.stream(cs):
            graph.replay()
        torch.cuda.synchronize()
        for j, t in enumerate(trips):
            want = _pass(eng, dev_tables, t, torch.randn((sizes[j], eng.Z), device=dev, generator=g))
            for k in want:
                assert_bits_equal(outs[j][k], want[k], f"replay {rep}, request {j}: {k}")
        assert eng.latent_stream() == (SEED, g.get_offset())


def test_host_ids_equals_the_device_pointer_form(cuda_models, dev_tables, synth, dev):
    import modular_prot_b_gan as m
    eng = m.make_fused_engine(*cuda_models)
    B = 3001
    trip = synth.make_triplets(B, seed=5)
    block = torch.zeros(3 * B, dtype=torch.float32).pin_memory()
    with pytest.raises(ValueError):
        eng.score_triplets_host_ids(*dev_tables, trip, block)          # needs the stream
    eng.set_latent_stream(True, SEED, 16)
    eng.score_triplets_host_ids(*dev_tables, trip, block)
    after = eng.latent_stream()
    eng.set_latent_stream(True, SEED, 16)
    want = _pass(eng, dev_tables, trip.to(dev), None, want_gen_scores=True, want_disc=True)
    assert eng.latent_stream() == after
    assert torch.equal(block[:B], want["gen_scores"].cpu())
    assert torch.equal(block[B:2 * B], want["logits"].cpu())
    assert torch.equal(block[2 * B:], want["probs"].cpu())
    bad = trip.clone()
    bad[7, 2] = 70000
    with pytest.raises(IndexError):
        eng.score_triplets_host_ids(*dev_tables, bad, block)
    eng.score_triplets_host_ids(*dev_tables, trip[:4].contiguous(), block[:12])   # the ctx is still healthy


# ----------------------------------------------------------------------------- modules and FusedInference
def test_generator_module_cuda_latents(dev, synth):
    import modular_prot_b_gan as m
    G, _ = synth.make_models(m.ModularGenerator, m.ModularDiscriminator)
    G = G.to(dev).eval()
    G.latent_source = "cuda"
    node_emb, rel_w = synth.make_tables(num_entities=4096)
    h, r = node_emb[:300].to(dev), rel_w[torch.arange(300) % 64].to(dev)
    g = twin(dev, m.LATENT_SEED)
    first = G(h, r)
    assert torch.equal(first, G(h, r, torch.randn((300, G.noise_dim), device=dev, generator=g)))
    z = G.sample_latent(10)
    assert z.device == dev and torch.equal(z, torch.randn((10, G.noise_dim), device=dev, generator=g))
    second = G(h, r)
    assert torch.equal(second, G(h, r, torch.randn((300, G.noise_dim), device=dev, generator=g)))
    assert not torch.equal(first, second)
    G.reseed()
    assert torch.equal(G(h, r), first)
    G.latent_source = "cpu"                              # the CPU stream is untouched by the device draws
    G.reseed(5)
    assert torch.equal(G.sample_latent(4), synth.make_latents(4, seed=5))


@pytest.fixture(scope="module")
def ckpt_path(tmp_path_factory, oracle, synth):
    path = tmp_path_factory.mktemp("ckpt") / "synthetic_ckpt.pt"
    torch.save(synth.make_checkpoint(oracle.ModularGenerator, oracle.ModularDiscriminator), path)
    return str(path)


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("bf16", 2e-2)])
def test_fused_inference_cuda_latents_match_the_oracle(ckpt_path, oracle_models, tables, synth, dev, precision, tol):
    import modular_prot_b_gan as m
    from pbg.inference import FusedInference
    inf = FusedInference(ckpt_path, "cuda", precision=precision, latents="cuda")
    Go, Do = oracle_models
    node_emb, rel_w = tables
    g = twin(dev, m.LATENT_SEED)
    for B in (5000, 17):
        trip = synth.make_triplets(B, seed=B)
        got = inf.score_triplets(json.dumps(trip.tolist()))
        z = torch.randn((B, 64), device=dev, generator=g).cpu()
        with torch.no_grad():
            h, r, t = node_emb[trip[:, 0]], rel_w[trip[:, 1]], node_emb[trip[:, 2]]
            gen = Go(h, r, z)
            cs, d = F.cosine_similarity(gen, t, dim=1), Do(h, r, t)
        scale = 1.0 if precision == "fp32" else max(d.abs().max().item(), 1.0)
        assert (torch.tensor(got["generator_scores"]) - cs).abs().max().item() <= tol
        assert (torch.tensor(got["discriminator_logits"]) - d).abs().max().item() <= tol * scale
        assert (torch.tensor(got["discriminator_probabilities"]) - torch.sigmoid(d)).abs().max().item() <= tol
    assert inf.engine.latent_stream()[1] == g.get_offset()
    # generator-only and discriminator-only requests, and predict_tails, use the same stream
    d_only = inf.score_triplets(trip.tolist(), method="discriminator")
    assert inf.engine.latent_stream()[1] == g.get_offset()
    assert d_only["discriminator_logits"] == got["discriminator_logits"]
    inf.reseed()
    a = inf.predict_tails(trip[:, :2].tolist(), top_k=5, return_scores=True)
    inf.reseed()
    assert inf.predict_tails(json.dumps(trip[:, :2].tolist()), top_k=5, return_scores=True) == a
    inf.reseed()
    b = inf.score_triplets(trip.tolist(), method="generator")
    inf.reseed()
    assert inf.score_triplets(trip.tolist())["generator_scores"] == b["generator_scores"]
