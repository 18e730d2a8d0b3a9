"""GPU parity tests (``-m gpu``): the CUDA path, called through the C ABI, against the CPU oracle on the same
seeded inputs.  Tolerances are the ones BASELINE.json's north_star states:
  fp32 mode : max-abs <= 1e-4           (config 2, B = 256)
  bf16 mode : relative error <= 2e-2    (config 3, B = 4096), rel = max|a-b| / max|b| per output tensor
  gather / index / sampling steps: bit-exact.
The oracle is builder-defined (the reference ships no model: parity is *unpinned*, see oracle header).
"""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

FP32_ATOL = 1e-4
BF16_REL = 2e-2


def rel_err(a: torch.Tensor, b: torch.Tensor) -> float:
    return ((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-12)).item()


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
def engine(cuda_models):
    import modular_prot_b_gan as m
    return m.make_fused_engine(*cuda_models)


@pytest.fixture(scope="module")
def dev_tables(tables, dev):
    node_emb, rel_w = tables
    return node_emb.to(dev), rel_w.to(dev)


def oracle_pass(oracle_models, tables, trip, z):
    Go, Do = oracle_models
    node_emb, rel_w = tables
    with torch.no_grad():
        h, r, t = node_emb[trip[:, 0]], rel_w[trip[:, 1]], node_emb[trip[:, 2]]
        g = Go(h, r, z)
        d = Do(h, r, t)
    return h, r, t, g, d, F.cosine_similarity(g, t, dim=1), torch.sigmoid(d)


# ----------------------------------------------------------------------------- config 2: fp32, B = 256
def test_fp32_b256_matches_oracle(engine, oracle_models, tables, dev_tables, synth, dev):
    B = 256
    trip, z = synth.make_triplets(B), synth.make_latents(B)
    _, _, _, g, d, cs, pr = oracle_pass(oracle_models, tables, trip, z)
    res = engine.score_triplets(*dev_tables, trip.to(dev), z.to(dev), want_gen_out=True, want_gen_scores=True,
                                want_disc=True, precision="fp32")
    engine.check_indices()
    assert res["gen_out"].shape == (B, 128) and res["gen_out"].dtype == torch.float32
    assert res["logits"].shape == (B,)
    assert (res["gen_out"].cpu() - g).abs().max().item() <= FP32_ATOL
    assert (res["logits"].cpu() - d).abs().max().item() <= FP32_ATOL
    assert (res["probs"].cpu() - pr).abs().max().item() <= FP32_ATOL
    assert (res["gen_scores"].cpu() - cs).abs().max().item() <= FP32_ATOL


# ----------------------------------------------------------------------------- config 3: bf16, B = 4096
def test_bf16_b4096_matches_oracle(engine, oracle_models, tables, dev_tables, synth, dev):
    B = 4096
    trip, z = synth.make_triplets(B), synth.make_latents(B)
    _, _, _, g, d, cs, pr = oracle_pass(oracle_models, tables, trip, z)
    res = engine.score_triplets(*dev_tables, trip.to(dev), z.to(dev), want_gen_out=True, want_gen_scores=True,
                                want_disc=True, precision="bf16")
    engine.check_indices()
    assert rel_err(res["gen_out"].cpu(), g) <= BF16_REL
    assert rel_err(res["logits"].cpu(), d) <= BF16_REL
    assert rel_err(res["probs"].cpu(), pr) <= BF16_REL
    assert rel_err(res["gen_scores"].cpu(), cs) <= BF16_REL
    # elementwise with an absolute floor: bf16 has 8 mantissa bits
    assert torch.allclose(res["gen_out"].cpu(), g, rtol=BF16_REL, atol=2e-2)


def test_bf16_output_dtype_bf16(engine, oracle_models, tables, dev_tables, synth, dev):
    B = 512
    trip, z = synth.make_triplets(B), synth.make_latents(B)
    _, _, _, g, *_ = oracle_pass(oracle_models, tables, trip, z)
    res = engine.score_triplets(*dev_tables, trip.to(dev), z.to(dev), want_gen_out=True, want_disc=False,
                                precision="bf16", out_dtype=torch.bfloat16)
    assert res["gen_out"].dtype == torch.bfloat16
    assert rel_err(res["gen_out"].float().cpu(), g) <= BF16_REL


# ----------------------------------------------------------------------------- per-layer known answers
@pytest.mark.parametrize("M", [1, 128, 200, 1000])
def test_tensor_core_layers_known_answer(engine, cuda_models, dev, M):
    """Each Linear of the PRODUCT kernel alone (pbg_linear_bf16 = the pass kernel with one item kind, its A operand the
    caller's matrix) against a torch fp32 product of the same bf16-rounded operands."""
    G, D = cuda_models
    gl = [(w.to(dev), b.to(dev)) for w, b in G.folded_layers()]
    dl = [(w.to(dev), b.to(dev)) for w, b in D.folded_layers()]
    torch.manual_seed(100 + M)

    def lin(a, w, b):
        return a.float() @ w.bfloat16().float().T + b

    a = (torch.randn(M, 320, device=dev) * 0.5).bfloat16()
    r0 = F.leaky_relu(lin(a, *gl[0]), 0.2)
    assert rel_err(eng_out := engine.linear_bf16(0, 0, a).float(), r0) <= 1e-2, "G layer 0"
    a1 = r0.bfloat16()
    r1 = F.leaky_relu(lin(a1, *gl[1]), 0.2)
    assert rel_err(engine.linear_bf16(0, 1, a1).float(), r1) <= 1e-2, "G layer 1"
    a2 = r1.bfloat16()
    r2 = torch.tanh(lin(a2, *gl[2]))
    assert (engine.linear_bf16(0, 2, a2) - r2).abs().max().item() <= 2e-3, "G layer 2 (tanh.approx)"
    d0 = (torch.randn(M, 384, device=dev) * 0.5).bfloat16()
    q0 = F.leaky_relu(lin(d0, *dl[0]), 0.2)
    assert rel_err(engine.linear_bf16(1, 0, d0).float(), q0) <= 1e-2, "D layer 0"
    d1 = q0.bfloat16()
    q1 = F.leaky_relu(lin(d1, *dl[1]), 0.2) @ dl[2][0].reshape(-1) + dl[2][1]
    assert (engine.linear_bf16(1, 1, d1) - q1).abs().max().item() <= 1e-3, "D layer 1 + folded final dot"
    del eng_out


# ----------------------------------------------------------------------------- bit-exact steps
def test_gather_is_bit_exact(engine, dev_tables, synth, dev):
    """forward-with-gather == forward on torch-gathered rows, bit for bit (fp32 mode: the only difference between the
    two calls is who performs the gather)."""
    B = 777
    trip, z = synth.make_triplets(B).to(dev), synth.make_latents(B).to(dev)
    node_emb, rel_w = dev_tables
    a = engine.generator_forward_gather(node_emb, rel_w, trip[:, 0], trip[:, 1], z, precision="fp32")
    b = engine.generator_forward(node_emb[trip[:, 0]], rel_w[trip[:, 1]], z, precision="fp32")
    assert torch.equal(a, b)
    a = engine.generator_forward_gather(node_emb, rel_w, trip[:, 0], trip[:, 1], z, precision="bf16")
    b = engine.generator_forward(node_emb[trip[:, 0]], rel_w[trip[:, 1]], z, precision="bf16")
    assert torch.equal(a, b)
    la = engine.score_triplets(node_emb, rel_w, trip, precision="fp32")["logits"]
    lb, _ = engine.discriminator_forward(node_emb[trip[:, 0]], rel_w[trip[:, 1]], node_emb[trip[:, 2]], precision="fp32")
    assert torch.equal(la, lb)


def test_latent_sampling_is_bit_exact(cuda_models, oracle_models):
    G, _ = cuda_models
    Go, _ = oracle_models
    G.reseed(99); Go.reseed(99)
    assert torch.equal(G.sample_latent(33), Go.sample_latent(33))
    G.reseed(); Go.reseed()


# ----------------------------------------------------------------------------- module boundary (SURVEY 8a/8b)
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("B", [1, 16, 127, 129, 255])
def test_module_boundary_ragged_batches(cuda_models, oracle_models, tables, synth, dev, B, prec):
    G, D = cuda_models
    G.precision = D.precision = prec
    try:
        trip, z = synth.make_triplets(B, seed=B), synth.make_latents(B, seed=B)
        h, r, t, g, d, _, pr = oracle_pass(oracle_models, tables, trip, z)
        node_emb, rel_w = tables
        out = G(h.to(dev), r.to(dev), z.to(dev))
        assert out.shape == (B, 128) and out.dtype == torch.float32 and out.is_contiguous()
        logits = D(h.to(dev), r.to(dev), t.to(dev))
        assert logits.dim() == 1 and logits.shape == (B,)  # 1-D: the REPL formats [0] with :.4f (:399-400)
        if B == 1:
            assert isinstance(logits.item(), float)  # pro_b_gan_infer.py:301
        rel_emb = torch.nn.Embedding(rel_w.shape[0], rel_w.shape[1]).to(dev)
        rel_emb.load_state_dict({"weight": rel_w})
        lg, pb = D.score_triplets(torch.nn.Parameter(node_emb.to(dev), requires_grad=False), rel_emb, trip.to(dev))
        if prec == "fp32":
            assert (out.cpu() - g).abs().max().item() <= FP32_ATOL
            assert (logits.cpu() - d).abs().max().item() <= FP32_ATOL
            assert (lg.cpu() - d).abs().max().item() <= FP32_ATOL
            assert (pb.cpu() - pr).abs().max().item() <= FP32_ATOL
        else:
            assert (out.cpu() - g).abs().max().item() <= BF16_REL * g.abs().max().item()
            assert (logits.cpu() - d).abs().max().item() <= BF16_REL * max(d.abs().max().item(), 0.05)
            assert (lg.cpu() - d).abs().max().item() <= BF16_REL * max(d.abs().max().item(), 0.05)
        assert len(lg.tolist()) == B and len(pb.tolist()) == B  # :208-209
    finally:
        G.precision = D.precision = None


def test_generator_draws_its_own_latents_like_the_oracle(cuda_models, oracle_models, tables, synth, dev):
    """forward(h, r) with no z: both modules draw from a CPU generator seeded 1234 (bit-exact sampling)."""
    G, _ = cuda_models
    Go, _ = oracle_models
    G.reseed(); Go.reseed()
    node_emb, rel_w = tables
    trip = synth.make_triplets(64)
    h, r = node_emb[trip[:, 0]], rel_w[trip[:, 1]]
    G.precision = "fp32"
    try:
        with torch.no_grad():
            ref = Go(h, r)
        out = G(h.to(dev), r.to(dev))
        assert (out.cpu() - ref).abs().max().item() <= FP32_ATOL
    finally:
        G.precision = None
        G.reseed(); Go.reseed()


def test_noncontiguous_index_columns(engine, dev_tables, synth, dev):
    """`triplet_tensor[:, i]` are stride-3 views (pro_b_gan_infer.py:183)."""
    trip = synth.make_triplets(300).to(dev)
    z = synth.make_latents(300).to(dev)
    node_emb, rel_w = dev_tables
    a = engine.generator_forward_gather(node_emb, rel_w, trip[:, 0], trip[:, 1], z, precision="fp32")
    b = engine.generator_forward_gather(node_emb, rel_w, trip[:, 0].contiguous(), trip[:, 1].contiguous(), z,
                                        precision="fp32")
    assert not trip[:, 0].is_contiguous()
    assert torch.equal(a, b)


def test_out_of_range_index_raises_indexerror(cuda_models, engine, dev_tables, synth, dev):
    """The CPU reference raises IndexError from `node_emb[heads]`; the CUDA path must too, without a sticky fault."""
    _, D = cuda_models
    node_emb, rel_w = dev_tables
    trip = synth.make_triplets(40).clone()
    trip[7, 2] = node_emb.shape[0] + 5
    rel_emb = torch.nn.Embedding(rel_w.shape[0], rel_w.shape[1]).to(dev)
    with pytest.raises(IndexError):
        D.score_triplets(node_emb, rel_emb, trip.to(dev))
    trip[7, 2] = 3
    trip[0, 1] = -1
    with pytest.raises(IndexError):
        D.score_triplets(node_emb, rel_emb, trip.to(dev))
    # the device is still healthy and the flag is cleared
    trip[0, 1] = 0
    D.score_triplets(node_emb, rel_emb, trip.to(dev))
    torch.cuda.synchronize()


def test_empty_batch(engine, dev_tables, dev):
    node_emb, rel_w = dev_tables
    res = engine.score_triplets(node_emb, rel_w, torch.empty(0, 3, dtype=torch.int64, device=dev),
                                torch.empty(0, 64, device=dev), want_gen_out=True, want_disc=True)
    assert res["gen_out"].shape == (0, 128) and res["logits"].shape == (0,)


def test_unloaded_model_and_cpu_module_fail_loudly(dev):
    import modular_prot_b_gan as m
    from pbg.engine import Engine
    from pbg.cabi import PbgError
    eng = Engine(128, 64, 1024, 1024, dev)
    with pytest.raises(PbgError):
        eng.discriminator_forward(torch.zeros(4, 128, device=dev), torch.zeros(4, 128, device=dev),
                                  torch.zeros(4, 128, device=dev))
    G = m.ModularGenerator(128, 64).eval()
    with pytest.raises(RuntimeError, match="no CPU path"):
        G(torch.zeros(2, 128), torch.zeros(2, 128))
    with pytest.raises(RuntimeError, match="inference-only"):
        m.ModularGenerator(128, 64).to(dev)(torch.zeros(2, 128, device=dev), torch.zeros(2, 128, device=dev))


# ----------------------------------------------------------------------------- host-buffer (end-to-end) entry point
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_host_entry_point_matches_device_entry_point(engine, dev_tables, synth, dev, prec):
    B = 1500
    trip, z = synth.make_triplets(B).pin_memory(), synth.make_latents(B).pin_memory()
    node_emb, rel_w = dev_tables
    gen = torch.empty(B, 128).pin_memory(); sc = torch.empty(B).pin_memory()
    lg = torch.empty(B).pin_memory(); pb = torch.empty(B).pin_memory()
    engine.score_triplets_host(node_emb, rel_w, trip, z, gen, sc, lg, pb, precision=prec)
    res = engine.score_triplets(node_emb, rel_w, trip.to(dev), z.to(dev), want_gen_out=True, want_gen_scores=True,
                                want_disc=True, precision=prec)
    assert torch.equal(gen, res["gen_out"].cpu()) and torch.equal(sc, res["gen_scores"].cpu())
    assert torch.equal(lg, res["logits"].cpu()) and torch.equal(pb, res["probs"].cpu())
    bad = trip.clone(); bad[3, 0] = 10 ** 9
    with pytest.raises(IndexError):
        engine.score_triplets_host(node_emb, rel_w, bad, z, gen, sc, lg, pb, precision=prec)


# ----------------------------------------------------------------------------- full-size, size-independent properties
def test_full_size_properties_b32768(engine, dev_tables, synth, dev):
    """BASELINE config 4 batch (32768) on one GPU: the oracle is too slow to be the checker at this size in a unit
    test, so check properties that hold for any correct batched row-wise map:
      * permutation equivariance: permuting the triplets permutes the outputs, bit for bit;
      * chunk invariance: the first 4096 rows of the big batch equal a 4096-row call, bit for bit;
      * duplicated rows give identical outputs; sigmoid(logit) == prob."""
    B = 32768
    trip, z = synth.make_triplets(B).to(dev), synth.make_latents(B).to(dev)
    trip[1] = trip[0]; z[1] = z[0]
    node_emb, rel_w = dev_tables
    kw = dict(want_gen_out=True, want_gen_scores=True, want_disc=True, precision="bf16")
    full = engine.score_triplets(node_emb, rel_w, trip, z, **kw)
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(5)).to(dev)
    shuf = engine.score_triplets(node_emb, rel_w, trip[perm], z[perm], **kw)
    for k in ("gen_out", "gen_scores", "logits", "probs"):
        assert torch.equal(full[k][perm], shuf[k]), k
    head = engine.score_triplets(node_emb, rel_w, trip[:4096], z[:4096], **kw)
    for k in ("gen_out", "gen_scores", "logits", "probs"):
        assert torch.equal(full[k][:4096], head[k]), k
    assert torch.equal(full["gen_out"][0], full["gen_out"][1]) and full["logits"][0] == full["logits"][1]
    assert torch.allclose(torch.sigmoid(full["logits"]), full["probs"], atol=1e-6)
    assert torch.isfinite(full["gen_out"]).all() and full["gen_out"].abs().max() <= 1.0


def test_batch_larger_than_one_chunk(engine, dev_tables, synth, dev):
    """Batches above the 65536-row workspace chunk are processed in pieces; results must not depend on it."""
    B = 65536 + 1000
    trip, z = synth.make_triplets(B).to(dev), synth.make_latents(B).to(dev)
    node_emb, rel_w = dev_tables
    full = engine.score_triplets(node_emb, rel_w, trip, z, want_gen_out=True, want_disc=True, precision="bf16")
    tail = engine.score_triplets(node_emb, rel_w, trip[65536:], z[65536:], want_gen_out=True, want_disc=True,
                                 precision="bf16")
    assert torch.equal(full["gen_out"][65536:], tail["gen_out"]) and torch.equal(full["logits"][65536:], tail["logits"])


# ----------------------------------------------------------------------------- launch width, lanes, result mirrors
def _pass(eng, dev_tables, trip, z, out=None):
    return eng.score_triplets(*dev_tables, trip, z, want_gen_out=True, want_gen_scores=True, want_disc=True,
                              precision="bf16", out_dtype=torch.bfloat16, out=out)


@pytest.mark.parametrize("B", [300, 4096, 9000])
def test_launch_width_does_not_change_a_single_bit(cuda_models, engine, dev_tables, synth, dev, B):
    """pbg_set_launch_width: the pass on 2, 48 or all SMs gives identical results (fixed-order reductions)."""
    import modular_prot_b_gan as m
    trip, z = synth.make_triplets(B).to(dev), synth.make_latents(B).to(dev)
    ref = {k: v.clone() for k, v in _pass(engine, dev_tables, trip, z).items()}
    for ctas in (2, 48, 74):
        eng = m.make_fused_engine(*cuda_models, ctas=ctas)
        res = _pass(eng, dev_tables, trip, z)
        eng.check_indices()
        for k in ref:
            assert torch.equal(res[k], ref[k]), f"width {ctas}: {k} differs"


@pytest.mark.parametrize("B", [31, 300, 4096, 9000])
def test_workspace_discard_does_not_change_a_single_bit(cuda_models, dev_tables, synth, dev, B):
    """pbg_set_workspace_discard: dropping dead activation / gathered row blocks from L2 (discard.global.L2) inside the pass
    changes no result -- same engine run repeatedly (a pass writes over what the previous one discarded), generator-only
    and discriminator-only passes, and a second engine with the option off as the reference."""
    import modular_prot_b_gan as m
    off, on = m.make_fused_engine(*cuda_models), m.make_fused_engine(*cuda_models)
    off.set_workspace_discard(False)
    on.set_workspace_discard(True)
    for rep in range(3):
        trip, z = synth.make_triplets(B, seed=700 + rep).to(dev), synth.make_latents(B, seed=800 + rep).to(dev)
        ref = {k: v.clone() for k, v in _pass(off, dev_tables, trip, z).items()}
        res = {k: v.clone() for k, v in _pass(on, dev_tables, trip, z).items()}
        for k in ref:
            assert torch.equal(res[k], ref[k]), f"rep {rep}: {k} differs with the discards on"
        for kw in (dict(want_gen_out=True, want_gen_scores=True, want_disc=False), dict(want_gen_out=False, want_gen_scores=False, want_disc=True)):
            a = off.score_triplets(*dev_tables, trip, z, precision="bf16", **kw)
            b = on.score_triplets(*dev_tables, trip, z, precision="bf16", **kw)
            for k in a:
                if a[k] is not None:
                    assert torch.equal(a[k], b[k]), f"rep {rep} {kw}: {k} differs with the discards on"
    off.check_indices(); on.check_indices()


def test_in_kernel_sm_clock_reading(cuda_models, dev_tables, synth, dev):
    """pbg_last_pass_sm_clock: clock64() ticks per globaltimer nanosecond over CTA 0's lifetime -- a plausible SM clock."""
    import modular_prot_b_gan as m
    eng = m.make_fused_engine(*cuda_models)
    trip, z = synth.make_triplets(4096).to(dev), synth.make_latents(4096).to(dev)
    for _ in range(3):
        _pass(eng, dev_tables, trip, z)
    mhz = eng.last_pass_sm_clock()
    assert 300.0 < mhz < 2500.0, mhz


def test_passes_on_concurrent_lanes_match_sequential(cuda_models, dev_tables, synth, dev):
    """Three ctxs on three streams, 48 SMs each, passes in flight together (bench.py's lanes)."""
    import modular_prot_b_gan as m
    B, S, R = 4096, 3, 4
    engines = [m.make_fused_engine(*cuda_models, ctas=48) for _ in range(S)]
    streams = [torch.cuda.Stream(dev) for _ in range(S)]
    inputs = [(synth.make_triplets(B, seed=100 + i).to(dev), synth.make_latents(B, seed=200 + i).to(dev)) for i in range(S * R)]
    ref = [{k: v.clone() for k, v in _pass(engines[0], dev_tables, t, z).items()} for t, z in inputs]
    torch.cuda.synchronize()
    got = []
    for i, (t, z) in enumerate(inputs):
        with torch.cuda.stream(streams[i % S]):
            got.append(_pass(engines[i % S], dev_tables, t, z))
    torch.cuda.synchronize()
    for e in engines:
        e.check_indices()
    for i in range(len(inputs)):
        for k in ref[i]:
            assert torch.equal(got[i][k], ref[i][k]), f"step {i}: {k} differs"


@pytest.mark.parametrize("B", [1000, 4096, 31])
def test_result_mirrors_receive_the_same_rows(cuda_models, dev_tables, synth, dev, B):
    """pbg_set_result_mirrors with two mirror buffers (same device here; peers' windows in a multi-GPU job).  The
    buffers carry 64 guard rows behind the batch: the bulk stores of a ragged last row group must not touch them."""
    import modular_prot_b_gan as m
    E, G = 128, 64
    eng = m.make_fused_engine(*cuda_models)
    trip, z = synth.make_triplets(B).to(dev), synth.make_latents(B).to(dev)
    mir = [{"gen_out": torch.full((B + G, E), 7.0, dtype=torch.bfloat16, device=dev), "gen_scores": torch.full((B + G,), 7.0, device=dev),
            "logits": torch.full((B + G,), 7.0, device=dev), "probs": torch.full((B + G,), 7.0, device=dev)} for _ in range(2)]
    eng.set_result_mirrors(**{k: [d[k].data_ptr() for d in mir] for k in mir[0]})
    res = _pass(eng, dev_tables, trip, z)
    torch.cuda.synchronize()
    for d in mir:
        for k in d:
            assert torch.equal(d[k][:B], res[k]), f"mirror {k} differs"
            assert bool((d[k][B:] == 7.0).all()), f"mirror {k}: rows behind the batch were written"
    with pytest.raises(Exception):   # mirrors are a bf16-mode feature: the fp32 path must refuse, not ignore them
        eng.score_triplets(*dev_tables, trip, z, want_gen_out=True, precision="fp32")
    eng.set_result_mirrors()
    res2 = _pass(eng, dev_tables, trip, z)
    assert torch.equal(res2["logits"], res["logits"])


# ----------------------------------------------------------------------------- BASELINE configs[4]: the width-scaled model
def test_wide_model_config5_matches_oracle(synth, dev):
    """E = 256, H = 4096 (SURVEY.md 8d's reading of "4x channels, 2x output resolution"), per-GPU batch 1024: the same
    pair kernel (biases through the global path: they no longer fit shared memory) against the fp32 oracle."""
    import modular_prot_b_gan as m
    from oracle import prot_b_gan_oracle as oracle
    E, Z, H, B, N = 256, 64, 4096, 1024, 8192
    Go, Do = synth.make_models(oracle.ModularGenerator, oracle.ModularDiscriminator, E, Z, H, H)
    G, D = synth.make_models(m.ModularGenerator, m.ModularDiscriminator, E, Z, H, H)
    node_emb, rel_w = synth.make_tables(N, 64, E)
    trip, z = synth.make_triplets(B, N, 64), synth.make_latents(B, Z)
    with torch.no_grad():
        h, r, t = node_emb[trip[:, 0]], rel_w[trip[:, 1]], node_emb[trip[:, 2]]
        g, d = Go(h, r, z), Do(h, r, t)
        cs = F.cosine_similarity(g, t, dim=1)
    eng = m.make_fused_engine(G.to(dev), D.to(dev))
    res = eng.score_triplets(node_emb.to(dev), rel_w.to(dev), trip.to(dev), z.to(dev), want_gen_out=True,
                             want_gen_scores=True, want_disc=True, precision="bf16")
    eng.check_indices()
    assert rel_err(res["gen_out"].cpu(), g) <= BF16_REL
    assert rel_err(res["logits"].cpu(), d) <= BF16_REL
    assert (res["probs"].cpu() - torch.sigmoid(d)).abs().max().item() <= BF16_REL
    assert (res["gen_scores"].cpu() - cs).abs().max().item() <= BF16_REL


# ----------------------------------------------------------------------------- staged requests (ingest / compute split)
@pytest.mark.parametrize("B", [1, 100, 4096, 5000])
def test_staged_request_equals_the_fused_pass_bit_for_bit(engine, dev_tables, synth, dev, B):
    """pbg_stage_triplets on an ingest stream + pbg_score_staged on the compute stream = pbg_score_triplets: the staging
    kernel copies the same rows with the same single bf16 rounding, the pass is the same kernel (gather phase off)."""
    trip, z = synth.make_triplets(B, seed=77).to(dev), synth.make_latents(B, seed=78).to(dev)
    ref = {k: v.clone() for k, v in _pass(engine, dev_tables, trip, z).items()}
    ingest = torch.cuda.Stream(dev)
    for slot in (0, 1):
        ingest.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(ingest):
            assert engine.stage_triplets(slot, *dev_tables, trip, z) == B
        torch.cuda.current_stream(dev).wait_stream(ingest)
        res = engine.score_staged(slot, want_gen_out=True, want_gen_scores=True, want_disc=True, out_dtype=torch.bfloat16)
        engine.check_indices()
        for k in ref:
            assert torch.equal(res[k], ref[k]), f"slot {slot}: {k} differs"


def test_staged_pipeline_in_a_cuda_graph_with_two_slots(cuda_models, dev_tables, synth, dev):
    """bench.py's lane: request j + 1 staged on the ingest stream while pass j runs, two slots, the whole sequence
    captured into one CUDA graph (pbg_reserve first: nothing may grow during capture) and replayed."""
    import modular_prot_b_gan as m
    B, n = 1000, 6
    eng = m.make_fused_engine(*cuda_models, ctas=48)
    inputs = [(synth.make_triplets(B, seed=300 + i).to(dev), synth.make_latents(B, seed=400 + i).to(dev)) for i in range(n)]
    ref = [{k: v.clone() for k, v in _pass(eng, dev_tables, t, z).items()} for t, z in inputs]
    outs = [{"gen_out": torch.zeros(B, 128, dtype=torch.bfloat16, device=dev), "gen_scores": torch.zeros(B, device=dev),
             "logits": torch.zeros(B, device=dev), "probs": torch.zeros(B, device=dev)} for _ in range(n)]
    fresh = m.make_fused_engine(*cuda_models, ctas=48)
    cs, ins = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(cs):
        with pytest.raises(Exception):          # growth inside a capture is refused, not a device-wide sync
            with torch.cuda.graph(torch.cuda.CUDAGraph(), stream=cs):
                fresh.stage_triplets(0, *dev_tables, *inputs[0])
    torch.cuda.synchronize()
    eng.reserve(B, "bf16", 2)
    with torch.cuda.stream(cs):
        with torch.cuda.graph(g, stream=cs):
            fork = torch.cuda.Event(); fork.record(cs); ins.wait_event(fork)
            done = [None, None]
            for j, (t, z) in enumerate(inputs):
                slot = j & 1
                with torch.cuda.stream(ins):
                    if done[slot] is not None:
                        ins.wait_event(done[slot])
                    eng.stage_triplets(slot, *dev_tables, t, z)
                    staged = torch.cuda.Event(); staged.record(ins)
                cs.wait_event(staged)
                eng.score_staged(slot, want_gen_out=True, want_gen_scores=True, want_disc=True, out_dtype=torch.bfloat16,
                                 out=outs[j])
                done[slot] = torch.cuda.Event(); done[slot].record(cs)
    for _ in range(3):
        for o in outs:
            for v in o.values():
                v.zero_()
        torch.cuda.synchronize()
        with torch.cuda.stream(cs):
            g.replay()
        torch.cuda.synchronize()
        for j in range(n):
            for k in ref[j]:
                assert torch.equal(outs[j][k], ref[j][k]), f"request {j}: {k} differs"
    eng.check_indices()


def test_pass_that_stages_the_next_request_equals_the_fused_pass(cuda_models, dev_tables, synth, dev):
    """pbg_score_staged_stage_next: pass j gathers request j + 1 into the other slot with its idle epilogue warps (same
    gather code as the fused pass, no arrivals, drained before exit).  A chain of ragged requests, bit for bit against
    the fused pass, eagerly and as one CUDA graph."""
    import modular_prot_b_gan as m
    sizes = [1000, 4096, 31, 257, 5000, 256, 3]
    eng = m.make_fused_engine(*cuda_models, ctas=48)
    inputs = [(synth.make_triplets(B, seed=700 + i).to(dev), synth.make_latents(B, seed=800 + i).to(dev)) for i, B in enumerate(sizes)]
    ref = [{k: v.clone() for k, v in _pass(eng, dev_tables, t, z).items()} for t, z in inputs]
    eng.reserve(max(sizes), "bf16", 2)
    kw = dict(want_gen_out=True, want_gen_scores=True, want_disc=True, out_dtype=torch.bfloat16)

    def chain(outs=None):
        res = []
        eng.stage_triplets(0, *dev_tables, *inputs[0])
        for j in range(len(inputs)):
            nxt = (*dev_tables, *inputs[j + 1]) if j + 1 < len(inputs) else None
            res.append(eng.score_staged(j & 1, stage_next=nxt, out=None if outs is None else outs[j], **kw))
        return res

    got = chain()
    torch.cuda.synchronize()
    eng.check_indices()
    for j in range(len(inputs)):
        for k in ref[j]:
            assert torch.equal(got[j][k], ref[j][k]), f"request {j} (B = {sizes[j]}): {k} differs"
    outs = [{k: torch.zeros_like(v) for k, v in r.items()} for r in ref]
    cs = torch.cuda.Stream(dev)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(cs):
        with torch.cuda.graph(g, stream=cs):
            chain(outs)
    for _ in range(2):
        for o in outs:
            for v in o.values():
                v.zero_()
        torch.cuda.synchronize()
        with torch.cuda.stream(cs):
            g.replay()
        torch.cuda.synchronize()
        for j in range(len(inputs)):
            for k in ref[j]:
                assert torch.equal(outs[j][k], ref[j][k]), f"graph, request {j}: {k} differs"
    # the stage-next form consumes its slot: scoring it again without staging it again is refused
    eng.stage_triplets(0, *dev_tables, *inputs[0])
    eng.score_staged(0, stage_next=(*dev_tables, *inputs[1]), **kw)
    with pytest.raises(Exception):
        eng.score_staged(0, **kw)
    eng.score_staged(1, **kw)            # the slot it staged is there, and a plain pbg_score_staged leaves it intact
    again = eng.score_staged(1, **kw)
    torch.cuda.synchronize()
    for k_ in ref[1]:
        assert torch.equal(again[k_], ref[1][k_]), f"slot scored twice: {k_} differs"
    # a bad id in the NEXT request is flagged by the pass that stages it
    bad = inputs[1][0].clone(); bad[3, 0] = 70000
    eng.stage_triplets(0, *dev_tables, *inputs[0])
    eng.score_staged(0, stage_next=(*dev_tables, bad, inputs[1][1]), **kw)
    with pytest.raises(IndexError):
        eng.check_indices()


def test_staged_request_flags_bad_ids_and_misuse(engine, dev_tables, synth, dev):
    B = 64
    z = synth.make_latents(B).to(dev)
    for col, bad in ((0, 65536), (1, -1), (2, -65537)):
        trip = synth.make_triplets(B).to(dev)
        trip[5, col] = bad
        engine.stage_triplets(0, *dev_tables, trip, z)
        engine.score_staged(0, want_disc=True)
        with pytest.raises(IndexError):
            engine.check_indices()
    trip = synth.make_triplets(B).to(dev)
    engine.stage_triplets(1, *dev_tables, trip, None, want_gen=False, want_disc=True)
    with pytest.raises(Exception):
        engine.score_staged(1, want_gen_out=True)           # no generator operands in the slot
    assert engine.score_staged(1, want_disc=True)["logits"].shape == (B,)
    engine.check_indices()


def test_generator_only_pass_still_validates_tail_ids(engine, dev_tables, synth, dev):
    """ADVICE r1: with no discriminator operand built nothing used to look at the tails; the reference raises
    IndexError at node_emb[tails] (pro_b_gan_infer.py:188) for every method."""
    B, N = 40, 65536
    z = synth.make_latents(B).to(dev)
    for prec in ("fp32", "bf16"):
        for bad in (N, -N - 1):
            trip = synth.make_triplets(B).to(dev)
            trip[7, 2] = bad
            engine.score_triplets(*dev_tables, trip, z, want_gen_scores=True, want_disc=False, precision=prec)
            with pytest.raises(IndexError):
                engine.check_indices()
        trip = synth.make_triplets(B).to(dev)
        trip[7, 2] = -1                                      # wraps to the last row, like tensor indexing
        a = engine.score_triplets(*dev_tables, trip, z, want_gen_scores=True, want_disc=False, precision=prec)
        trip[7, 2] = N - 1
        b = engine.score_triplets(*dev_tables, trip, z, want_gen_scores=True, want_disc=False, precision=prec)
        engine.check_indices()
        assert torch.equal(a["gen_scores"], b["gen_scores"])


# ----------------------------------------------------------------------------- stress: the relaxed layer hand-off
def test_stress_ragged_sizes_on_concurrent_lanes_bit_identical(cuda_models, dev_tables, synth, dev):
    """>= 200 passes over ragged batch sizes on 3 concurrent lanes (48 SMs each, as bench.py runs them), every result
    compared bit for bit with the first run of its inputs: the activation hand-off (bulk-store completion + relaxed
    counter increment, consumer's relaxed poll + proxy fence, DESIGN.md 3.1) has no other check than this -- a missed
    dependency shows as a mismatch, a lost arrival as a hang (the in-kernel guard traps)."""
    import modular_prot_b_gan as m
    S = 3
    sizes = [1, 31, 255, 256, 257, 1000, 4096, 5000, 9000]
    engines = [m.make_fused_engine(*cuda_models, ctas=48) for _ in range(S)]
    streams = [torch.cuda.Stream(dev) for _ in range(S)]
    inputs = [(synth.make_triplets(B, seed=500 + i).to(dev), synth.make_latents(B, seed=600 + i).to(dev)) for i, B in enumerate(sizes)]
    ref = [{k: v.clone() for k, v in _pass(engines[0], dev_tables, t, z).items()} for t, z in inputs]
    torch.cuda.synchronize()
    n = 0
    for rep in range(8):
        got = []
        for i in range(3 * len(sizes)):
            j = (i * 7 + rep) % len(sizes)
            with torch.cuda.stream(streams[i % S]):
                got.append((j, _pass(engines[i % S], dev_tables, *inputs[j])))
        torch.cuda.synchronize()
        for j, res in got:
            n += 1
            for k in ref[j]:
                assert torch.equal(res[k], ref[j][k]), f"rep {rep}, B = {sizes[j]}: {k} differs"
    for e in engines:
        e.check_indices()
    assert n >= 200


# ----------------------------------------------------------------------------- host entry points
@pytest.mark.parametrize("B", [4096, 333])
def test_host_entry_points_packed_and_per_buffer(engine, dev_tables, synth, dev, B):
    """pbg_score_triplets_host_packed moves [triplets | z] and [scores | logits | probs] in one copy each (an odd B: z is
    not 16-byte aligned behind the triplets, the inputs go in two copies); pbg_score_triplets_host copies buffer by
    buffer.  Same results either way, equal to the device-pointer call."""
    trip, z = synth.make_triplets(B, seed=31), synth.make_latents(B, seed=32)
    ref = _pass(engine, dev_tables, trip.to(dev), z.to(dev))
    blk = torch.empty(B * (24 + 64 * 4), dtype=torch.uint8).pin_memory()
    blk[:B * 24].view(torch.int64).view(B, 3).copy_(trip)
    blk[B * 24:].view(torch.float32).view(B, 64).copy_(z)
    hb = torch.zeros(3 * B).pin_memory()
    engine.score_triplets_host_packed(*dev_tables, blk, hb, B, precision="bf16")
    sep = [torch.zeros(B).pin_memory() for _ in range(3)]
    gen = torch.zeros(B, 128).pin_memory()
    engine.score_triplets_host(*dev_tables, trip.clone().pin_memory(), z.clone().pin_memory(), gen, *sep, precision="bf16")
    for i, k in enumerate(("gen_scores", "logits", "probs")):
        assert torch.equal(hb[i * B:(i + 1) * B], ref[k].cpu()), k
        assert torch.equal(sep[i], ref[k].cpu()), k
    assert torch.equal(gen.bfloat16(), ref["gen_out"].cpu())   # the host form returns fp32 rows of the same values
    with pytest.raises(ValueError):
        engine.score_triplets_host_packed(*dev_tables, blk[:-8], hb, B)


def test_bench_dump_outputs_are_the_last_timed_steps_results(synth, dev, tmp_path):
    """bench.py --dump-outputs on the B200 arm: the last of K timed steps ran pool entry K - 1 (K below the pool size);
    its dumped rows equal, bit for bit, a direct fused pass over that entry's seeded inputs."""
    import importlib.util
    import subprocess
    import sys
    from pathlib import Path
    import numpy as np
    import modular_prot_b_gan as m
    root = Path(__file__).resolve().parent.parent
    K = 20
    out = subprocess.run([sys.executable, str(root / "bench.py"), "--steps", str(K), "--warmup", "3", "--trials", "1",
                          "--no-cpu-baseline", "--no-library-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    spec = importlib.util.spec_from_file_location("bench_mod", str(root / "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    cfg = bench.CONFIGS["base"]
    B = cfg["batch"]
    G, D = bench.make_models(cfg, m.ModularGenerator, m.ModularDiscriminator)
    eng = m.make_fused_engine(G.to(dev), D.to(dev))
    node_emb, rel_w = (t.to(dev) for t in synth.make_tables(bench.NUM_ENTITIES, bench.NUM_RELATIONS, cfg["E"]))
    trip = synth.make_triplets(B, bench.NUM_ENTITIES, bench.NUM_RELATIONS, seed=4321 + K - 1).to(dev)
    z = synth.make_latents(B, cfg["Z"], seed=1234 + K - 1).to(dev)
    ref = eng.score_triplets(node_emb, rel_w, trip, z, want_gen_out=True, want_gen_scores=True, want_disc=True,
                             precision="bf16", out_dtype=torch.bfloat16)
    torch.cuda.synchronize()
    assert sorted(p.name for p in tmp_path.iterdir()) == ["gen_out.npy", "gen_scores.npy", "logits.npy", "probs.npy"]
    for k in ("gen_out", "gen_scores", "logits", "probs"):
        got = np.load(tmp_path / f"{k}.npy")
        assert got.dtype == np.float32, k
        assert np.array_equal(got, ref[k].float().cpu().numpy()), k
