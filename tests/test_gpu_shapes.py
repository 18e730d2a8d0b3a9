"""The fused pass and the fp32 path at model shapes that select each of their branches.

``pbg_create`` accepts any embed_dim / noise_dim / g_hidden that are multiples of 8, any d_hidden that is a multiple of
16 and any leaky_slope in [0, 1], and the shape decides which code runs: first-layer K padding, padded hidden widths,
the pass instance (FASTG, BIASS), 128- or 256-wide tiles, how the generator's last layer reduces its cosine and stores
its rows, and the partial-buffer limits.  ``branches()`` restates the host's selection formulas, ``SHAPES`` is a small
matrix that reaches both values of every flag, and the checks run each shape against a float64 reference that rounds
to bf16 exactly where the kernels round:

  A  each tensor-core layer alone (pbg_linear_bf16) on the reference's own bf16 operands, within an error bound
  B  the fused pass equals the chain of single-layer launches bit for bit
  C  the fused bf16 pass against the unrounded float64 model (relative error 2e-2)
  D  fp32 mode against the float64 model (1e-4)
  E  bit-exact invariants of the bf16 pass: G-only / D-only passes, staging, stage-next, launch width, result
     mirrors, the trace instance
  F  the dims pbg_create refuses, and the bf16-mode limits (embed_dim <= 512 with the generator, d_hidden <= 8192)

The tests without the gpu marker check the harness itself on the CPU: the branch map of the matrix, the reference
against the oracle modules, its bf16 rounding, and that check A's bound rejects a dropped K block or output chunk.
Only one engine (one pbg_ctx) is alive at a time.
"""
import copy
import functools
import gc

import numpy as np
import pytest
import torch

# --------------------------------------------------------------------------------------------- the shape matrix
# id: (embed_dim E, noise_dim Z, g_hidden HG, d_hidden HD, leaky_slope)
SHAPES = {
    "S0": (128, 64, 1024, 1024, 0.2),   # today's shape: FASTG, BIASS, in_cta, pair_out
    "S1": (128, 32, 1000, 1008, 0.01),  # K 288 -> 320 (FASTG off), HG 1000 / HD 1008 -> 1024, H/2 504 -> 512
    "S2": (64, 16, 256, 128, 0.2),      # K 144 -> 192, in_cta with the upper chunk padding, D tiles 128 wide
    "S3": (8, 8, 8, 16, 0.0),           # every width padded, n_valid = 8, ReLU
    "S4": (192, 64, 2048, 2048, 0.2),   # one G L2 tile of 4 chunks (chunk 3 padding); BIASS off only for the full pass
    "S5": (200, 24, 1536, 1552, 0.5),   # K padding on both models, HD 1552 -> 1664, H/2 776 -> 896, 128-wide tiles
    "S6": (320, 64, 1024, 1024, 0.2),   # G L2 over 3 tiles of 128 (partials across tiles)
    "S7": (512, 64, 4096, 8192, 0.2),   # the limits: slots_g = 8, slots_d = 64
    "S8": (128, 128, 2048, 2048, 0.2),  # FASTG with BIASS off for the full pass (8320 bias floats), Z = 128
}
SHAPE_IDS = list(SHAPES)
# shapes beyond the bf16-mode limits (check F)
LIMIT_E = (520, 8, 64, 64, 0.2)       # G L2 needs 10 cosine partial slots, the buffer holds 8
LIMIT_HD = (128, 64, 64, 8208, 0.2)   # D L1 needs 66 dot partial slots (H/2 = 4104 -> 4224), the buffer holds 64

N_ENT, N_REL = 4096, 64


def batches(sid):
    """One row, fewer than the 32 rows of pair_out, one row past a 256-row block, a ragged fourth block."""
    return (1, 31, 257, 1000) + ((4096,) if sid in ("S0", "S1", "S8") else ())


# --------------------------------------------------------------------------------------------- the branch map
BIAS_SMEM_FLOATS = 6144   # P2Smem::kBiasFloats (pass2_kernel.cuh)
SLOTS_G_MAX = 8           # kPartSlotsG / 2 (pbg.cu)
SLOTS_D_MAX = 64          # kPartSlotsD (pbg.cu)


def round_up(v, m):
    return (v + m - 1) // m * m


def branches(E, Z, HG, HD):
    """The host's selection formulas, restated from csrc/pbg.cu:
      pbg_create (kg0p, kd0p, hgp, hdp) and upload_linear (np = round_up(n, 128));
      set_layer (block_n: 256 when np % 256 == 0, else 128);
      launch_pass2: biass (sum of the padded biases of the layers on, + D L1's np for w3, <= kBiasFloats), the slot
      limits (np / 64 of D L1 <= kPartSlotsD, of G L2 <= kPartSlotsG / 2), slots_g, slots_d and fastg;
    and from the PEPI_TANH epilogue of pass2_kernel.cuh: in_cta, pair_out (bf16 out) and bulk_mirror."""
    kg0, kd0 = 2 * E + Z, 3 * E
    kg0p, kd0p = round_up(kg0, 64), round_up(kd0, 64)
    hgp, hdp = round_up(HG, 128), round_up(HD, 128)
    np_ = {"g0": hgp, "d0": hdp, "g1": hgp, "d1": round_up(HD // 2, 128), "g2": round_up(E, 128)}
    kp = {"g0": kg0p, "d0": kd0p, "g1": hgp, "d1": hdp, "g2": hgp}
    block_n = {k: 256 if v % 256 == 0 else 128 for k, v in np_.items()}
    n_tiles = {k: np_[k] // block_n[k] for k in np_}

    def biass(g, d):
        floats = (np_["g0"] + np_["g1"] + np_["g2"] if g else 0) + (np_["d0"] + 2 * np_["d1"] if d else 0)
        return floats <= BIAS_SMEM_FLOATS

    in_cta = n_tiles["g2"] == 1 and block_n["g2"] == 128
    return dict(
        kg0=kg0, kd0=kd0, kg0p=kg0p, kd0p=kd0p, hgp=hgp, hdp=hdp, np=np_, kp=kp, block_n=block_n, n_tiles=n_tiles,
        bias_floats_full=np_["g0"] + np_["g1"] + np_["g2"] + np_["d0"] + 2 * np_["d1"],
        fastg=E == 128 and Z % 4 == 0 and Z <= 128 and kg0p == kg0 and kd0p == kd0,
        biass_full=biass(True, True), biass_g=biass(True, False), biass_d=biass(False, True),
        in_cta=in_cta, pair_out=in_cta and E == 128, bulk_mirror=E % 64 == 0,
        slots_g=(E + 63) // 64, slots_d=np_["d1"] // 64,
        g_ok=np_["g2"] // 64 <= SLOTS_G_MAX, d_ok=np_["d1"] // 64 <= SLOTS_D_MAX)


def flags(E, Z, HG, HD):
    """The two-valued branch flags of one shape."""
    b = branches(E, Z, HG, HD)
    return {
        "k_pad_g": b["kg0p"] != b["kg0"], "k_pad_d": b["kd0p"] != b["kd0"],
        "hg_pad": b["hgp"] != HG, "hd_pad": b["hdp"] != HD, "d1_pad": b["np"]["d1"] != HD // 2,
        "fastg": b["fastg"], "biass_full": b["biass_full"],
        "biass_differs_g_or_d_only": b["biass_full"] != b["biass_g"] or b["biass_full"] != b["biass_d"],
        "tiles128_not_g2": any(b["block_n"][k] == 128 for k in ("g0", "d0", "g1", "d1")),
        "in_cta": b["in_cta"], "pair_out": b["pair_out"], "g2_tiles_gt1": b["n_tiles"]["g2"] > 1,
        "g2_ragged": E % 64 != 0, "bulk_mirror": b["bulk_mirror"], "upper_chunk_padding": b["np"]["g2"] - E >= 64,
    }


def accepted(E, Z, HG, HD, slope):
    """The dims pbg_create accepts (pbg.cu: pbg_create)."""
    return min(E, Z, HG, HD) > 0 and E % 8 == 0 and Z % 8 == 0 and HG % 8 == 0 and HD % 16 == 0 and 0.0 <= slope <= 1.0


def test_branch_map_matrix_reaches_every_branch():
    assert all(accepted(*d) for d in (*SHAPES.values(), LIMIT_E, LIMIT_HD))
    per = {sid: flags(*SHAPES[sid][:4]) for sid in SHAPE_IDS}
    for name in per["S0"]:
        seen = {per[sid][name] for sid in SHAPE_IDS}
        assert seen == {True, False}, f"{name}: the matrix only reaches {seen}"
    br = {sid: branches(*SHAPES[sid][:4]) for sid in SHAPE_IDS}
    assert max(b["slots_g"] for b in br.values()) == SLOTS_G_MAX and all(b["g_ok"] for b in br.values())
    assert max(b["slots_d"] for b in br.values()) == SLOTS_D_MAX and all(b["d_ok"] for b in br.values())
    assert {s for (*_, s) in SHAPES.values()} >= {0.0, 0.01, 0.2, 0.5}
    assert not branches(*LIMIT_E[:4])["g_ok"] and branches(*LIMIT_E[:4])["d_ok"]
    assert branches(*LIMIT_HD[:4])["g_ok"] and not branches(*LIMIT_HD[:4])["d_ok"]
    # the values the matrix was chosen for
    assert (br["S1"]["kg0p"], br["S1"]["hgp"], br["S1"]["np"]["d1"]) == (320, 1024, 512)
    assert (br["S5"]["kg0p"], br["S5"]["kd0p"], br["S5"]["hdp"], br["S5"]["np"]["d1"]) == (448, 640, 1664, 896)
    assert br["S5"]["block_n"]["d0"] == br["S5"]["block_n"]["d1"] == 128
    assert br["S8"]["bias_floats_full"] == 8320 and br["S8"]["fastg"] and br["S8"]["biass_g"]
    assert not br["S4"]["biass_full"] and br["S4"]["biass_g"] and br["S4"]["biass_d"]
    assert br["S6"]["n_tiles"]["g2"] == 3 and br["S4"]["n_tiles"]["g2"] == 1 and br["S4"]["block_n"]["g2"] == 256


# --------------------------------------------------------------------------------------------- the reference
def bf16(x):
    """Round to bf16 (round to nearest even), keeping the dtype."""
    return x.to(torch.bfloat16).to(x.dtype)


def leaky(x, slope):
    return torch.where(x >= 0, x, x * slope)


def fold64(lin, bn):
    """pbg.engine.fold_linear_bn without its final rounding to fp32 (for the comparison with the float64 oracle)."""
    W, b = lin.weight.detach().double(), lin.bias.detach().double()
    if bn is not None:
        s = bn.weight.detach().double() / torch.sqrt(bn.running_var.detach().double() + bn.eps)
        W, b = W * s[:, None], (b - bn.running_mean.detach().double()) * s + bn.bias.detach().double()
    return W, b


def fold_models(G, D, fold):
    """[(W, b)] * 3 for G and for D, BatchNorm folded by `fold` (pbg.engine.fold_linear_bn for the engine)."""
    g, d = G.net, D.net
    return ([fold(g[0], g[1]), fold(g[3], g[4]), fold(g[6], None)],
            [fold(d[0], None), fold(d[2], None), fold(d[4], None)])


class RefModel:
    """The folded weights as float64, zero-padded to the kernels' [Np, Kp] grid; rounded to bf16 when `rnd` (biases and
    the final dot weights stay as they are: the kernels read them as fp32)."""

    def __init__(self, dims, g_layers, d_layers, rnd, device):
        E, Z, HG, HD, self.slope = dims
        self.E, self.rnd = E, rnd
        b = branches(E, Z, HG, HD)
        self.kg0p, self.kd0p = b["kg0p"], b["kd0p"]

        def pad(W, bias, key):
            W = W.double()
            Wp = torch.zeros(b["np"][key], b["kp"][key], dtype=torch.float64)
            Wp[:W.shape[0], :W.shape[1]] = bf16(W) if rnd else W
            bp = torch.zeros(b["np"][key], dtype=torch.float64)
            bp[:bias.shape[0]] = bias.double()
            return Wp.to(device), bp.to(device), W.shape[0], W.shape[1]

        self.g = [pad(*g_layers[0], "g0"), pad(*g_layers[1], "g1"), pad(*g_layers[2], "g2")]
        self.d = [pad(*d_layers[0], "d0"), pad(*d_layers[1], "d1")]
        w3 = torch.zeros(b["np"]["d1"], dtype=torch.float64)
        w3[:HD // 2] = d_layers[2][0].reshape(-1).double()
        self.w3, self.b3 = w3.to(device), float(d_layers[2][1].reshape(-1)[0])

    def q(self, x):
        return bf16(x) if self.rnd else x

    def inputs(self, node_emb, rel_w, trip, z):
        """First-layer inputs [h | r | z | 0...] and [h | r | t | 0...] (node_emb[-i] wraps like the gather)."""
        h, r, t = node_emb[trip[:, 0]].double(), rel_w[trip[:, 1]].double(), node_emb[trip[:, 2]].double()
        xg = torch.cat([h, r, z.double()], 1)
        xd = torch.cat([h, r, t], 1)
        xg = torch.nn.functional.pad(xg, (0, self.kg0p - xg.shape[1]))
        xd = torch.nn.functional.pad(xd, (0, self.kd0p - xd.shape[1]))
        return self.q(xg), self.q(xd), t

    # the epilogues, from the pre-activation x @ W^T
    def store(self, pre, layer):
        return self.q(leaky(pre + layer[1], self.slope))

    def rowdot(self, pre, layer):
        return leaky(pre + layer[1], self.slope) @ self.w3 + self.b3

    def tanh(self, pre, layer):
        return torch.tanh(pre + layer[1])[:, :self.E]

    def forward(self, xg, xd):
        """The layer outputs of G (g0, g1, gen) and D (d0, logit)."""
        g0 = self.store(xg @ self.g[0][0].T, self.g[0])
        g1 = self.store(g0 @ self.g[1][0].T, self.g[1])
        gen = self.tanh(g1 @ self.g[2][0].T, self.g[2])
        d0 = self.store(xd @ self.d[0][0].T, self.d[0])
        logit = self.rowdot(d0 @ self.d[1][0].T, self.d[1])
        return g0, g1, gen, d0, logit


def cosine64(g, t):
    """F.cosine_similarity(g, t, dim=1) with eps 1e-8 on each norm, in float64."""
    g, t = g.double(), t.double()
    return (g * t).sum(1) / (g.norm(dim=1).clamp_min(1e-8) * t.norm(dim=1).clamp_min(1e-8))


# --------------------------------------------------------------------------------------------- check A's bound
ACC = 2.0 ** -14   # accumulation term per unit of sum_k |a_k w_k|
TANH_ATOL = 2e-3   # tanh.approx in the G L2 epilogue (as test_tensor_core_layers_known_answer)


def ulp_bf16(v):
    """One bf16 ulp of |v| (0 for v = 0)."""
    _, e = torch.frexp(v.abs())
    return torch.where(v != 0, torch.pow(2.0, (e - 8).to(v.dtype)), torch.zeros_like(v))


def ratio(err, bound):
    """Largest err / bound (inf where the bound is 0 and the error is not)."""
    r = torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err > 0, float("inf"), 0.0))
    return r.max().item() if r.numel() else 0.0


def bound_store(ref, a, W):
    return ulp_bf16(ref) + ACC * (a.abs() @ W.abs().T)


def bound_rowdot(a, W, b, w3, slope):
    """The accumulation term of every hidden column, carried through the LeakyReLU (which scales the error of a column
    that is negative beyond its own error by the slope) and the final dot with w3."""
    e = ACC * (a.abs() @ W.abs().T)
    y = a @ W.T + b
    return (torch.where(y < -e, slope * e, e)) @ w3.abs()


@functools.lru_cache(maxsize=1)
def cpu_models(dims):
    from oracle import prot_b_gan_oracle as oracle
    from pbg import synth
    E, Z, HG, HD, _ = dims
    return synth.make_models(oracle.ModularGenerator, oracle.ModularDiscriminator, E, Z, HD, g_hidden=HG)


def sample(B, Z, seed):
    """Triplets over N_ENT x N_REL with negative head (every 3rd row) and tail (every 4th) ids, and latents."""
    from pbg import synth
    trip = synth.make_triplets(B, N_ENT, N_REL, seed=seed)
    trip[0::3, 0] -= N_ENT
    trip[1::4, 2] -= N_ENT
    return trip, synth.make_latents(B, Z, seed=seed + 1)


# --------------------------------------------------------------------------------------------- CPU tests of the harness
@pytest.mark.parametrize("sid", ["S2", "S3"])
def test_reference_without_rounding_equals_the_oracle(sid):
    from oracle import prot_b_gan_oracle as oracle
    from pbg import synth
    E, Z, HG, HD, _ = SHAPES[sid]
    dims = (E, Z, HG, HD, oracle.LEAKY_SLOPE)
    G, D = cpu_models(dims)
    ref = RefModel(dims, *fold_models(G, D, fold64), rnd=False, device="cpu")
    node_emb, rel_w = synth.make_tables(N_ENT, N_REL, E)
    trip, z = sample(300, Z, seed=5)
    xg, xd, t = ref.inputs(node_emb, rel_w, trip, z)
    _, _, gen, _, logit = ref.forward(xg, xd)
    with torch.no_grad():
        G64, D64 = copy.deepcopy(G).double(), copy.deepcopy(D).double()
        h, r = node_emb[trip[:, 0]].double(), rel_w[trip[:, 1]].double()
        g_want, d_want = G64(h, r, z.double()), D64(h, r, t)
    assert (gen - g_want).abs().max().item() <= 1e-10
    assert (logit - d_want).abs().max().item() <= 1e-10


def test_reference_bf16_rounding_is_round_to_nearest_even():
    """The reference rounds float64 values that fp32 holds exactly (inputs, weights) and float64 sums: both must land
    where torch's own fp32 -> bf16 conversion (and the kernels' __float2bfloat16_rn) does.  Checked against an integer
    round-to-nearest-even of the fp32 bit patterns, ties and near-ties included."""
    g = torch.Generator().manual_seed(11)
    bits = torch.randint(0, 2 ** 31 - 1, (200000,), generator=g, dtype=torch.int64)
    bits = torch.cat([bits, (bits & ~0xFFFF) | 0x8000, (bits & ~0xFFFF) | 0x7FFF, (bits & ~0xFFFF) | 0x8001])
    bits = torch.cat([bits, bits | (1 << 31)])                      # both signs
    bits = bits[((bits >> 23) & 0xFF) != 0xFF]                       # no inf / NaN
    as_f32 = lambda u: torch.from_numpy(u.numpy().astype(np.uint32).view(np.float32))
    x32 = as_f32(bits)
    want = as_f32(((bits + 0x7FFF + ((bits >> 16) & 1)) >> 16) << 16)
    assert torch.equal(x32.bfloat16().float(), want)
    assert torch.equal(bf16(x32.double()), want.double())
    assert torch.equal(bf16(x32), want)


def _layer_cases(sid, rows=256):
    """(name, a, layer, epilogue) of every layer of shape `sid` on the CPU, with its operands from the rounded
    reference chain."""
    from pbg import engine as pbg_engine
    from pbg import synth
    dims = SHAPES[sid]
    E, Z = dims[:2]
    ref = RefModel(dims, *fold_models(*cpu_models(dims), pbg_engine.fold_linear_bn), rnd=True, device="cpu")
    node_emb, rel_w = synth.make_tables(N_ENT, N_REL, E)
    xg, xd, _ = ref.inputs(node_emb, rel_w, *sample(rows, Z, seed=9))
    g0, g1, _, d0, _ = ref.forward(xg, xd)
    return ref, [("G L0", xg, ref.g[0], ref.store), ("G L1", g0, ref.g[1], ref.store), ("G L2", g1, ref.g[2], ref.tanh),
                 ("D L0", xd, ref.d[0], ref.store), ("D L1", d0, ref.d[1], ref.rowdot)]


def _bound(want, a, layer, epi, ref):
    """Check A's tolerance of one layer output."""
    if epi == ref.tanh:
        return torch.full_like(want, TANH_ATOL)
    if epi == ref.rowdot:
        return bound_rowdot(a, layer[0], layer[1], ref.w3, ref.slope)
    return bound_store(want, a, layer[0])


@pytest.mark.parametrize("sid", SHAPE_IDS)
def test_check_a_bound_rejects_a_dropped_k_block_or_output_chunk(sid):
    """Check A's tolerance is tight enough to see the bugs that padding and tiling produce: a kernel that skipped any one
    64-wide K block holding real columns, or zeroed any one 64-column output chunk holding real columns, fails it at
    every shape -- and a correct product accumulated differently (fp32, another order) passes it."""
    ref, cases = _layer_cases(sid)
    for name, a, layer, epi in cases:
        W, n_real, k_real = layer[0], layer[2], layer[3]
        pre = a @ W.T
        want = epi(pre, layer)
        bound = _bound(want, a, layer, epi, ref)
        within = lambda got: bool(((got - want).abs() <= bound).all())
        assert within(epi((a.float() @ W.float().T).double(), layer)), f"{sid} {name}: a correct fp32 product fails"
        for kb in range(0, k_real, 64):   # the K blocks past the real columns are padding: leaving them out is no bug
            dropped = epi(pre - a[:, kb:kb + 64] @ W[:, kb:kb + 64].T, layer)
            assert not within(dropped), f"{sid} {name}: K block {kb // 64} dropped, bound holds"
        for c0 in range(0, n_real, 64):   # likewise the output chunks
            if epi == ref.rowdot:
                h = leaky(pre + layer[1], ref.slope)
                zeroed = want - h[:, c0:c0 + 64] @ ref.w3[c0:c0 + 64]
            else:
                zeroed = want.clone()
                zeroed[:, c0:c0 + 64] = 0
            assert not within(zeroed), f"{sid} {name}: chunk {c0 // 64} zeroed, bound holds"


# --------------------------------------------------------------------------------------------- GPU: one engine at a time
_live = []   # [(owner, Engine)]: the one engine of this module that may be alive, and its only lasting reference


def _free_engine():
    _live.clear()
    gc.collect()
    if torch.cuda.is_available():
        torch.cuda.synchronize()


def make_engine(dims, g_layers, d_layers, dev, owner=None):
    """A plain Engine(E, Z, HG, HD, dev, leaky_slope) with the folded weights loaded, after freeing any other."""
    from pbg.engine import Engine
    _free_engine()
    E, Z, HG, HD, slope = dims
    eng = Engine(E, Z, HG, HD, dev, leaky_slope=slope)
    if g_layers is not None:
        eng.load_generator(g_layers)
    if d_layers is not None:
        eng.load_discriminator(d_layers)
    _live.append((owner, eng))
    return eng


class Case:
    """One shape: its weights, float64 references (rounded and not) and tables on the device, and its engine."""

    def __init__(self, dims, dev):
        from pbg import engine as pbg_engine
        from pbg import synth
        self.dims, self.dev = dims, dev
        self.E, self.Z = dims[:2]
        self.g_layers, self.d_layers = fold_models(*cpu_models(dims), pbg_engine.fold_linear_bn)
        self.ref = RefModel(dims, self.g_layers, self.d_layers, rnd=True, device=dev)
        self.exact = RefModel(dims, self.g_layers, self.d_layers, rnd=False, device=dev)
        node_emb, rel_w = synth.make_tables(N_ENT, N_REL, self.E)
        self.node_emb, self.rel_w = node_emb.to(dev), rel_w.to(dev)

    @property
    def eng(self):
        """This shape's engine, (re)made when another one has taken its place."""
        if _live and _live[0][0] is self:
            return _live[0][1]
        return make_engine(self.dims, self.g_layers, self.d_layers, self.dev, owner=self)

    def sample(self, B):
        trip, z = sample(B, self.Z, seed=1000 + B)
        return trip.to(self.dev), z.to(self.dev)

    def run(self, trip, z, precision="bf16", out_dtype=torch.float32, gen=True, disc=True, **kw):
        return self.eng.score_triplets(self.node_emb, self.rel_w, trip, z, want_gen_out=gen, want_gen_scores=gen,
                                       want_disc=disc, precision=precision, out_dtype=out_dtype, **kw)

    def close(self):
        if _live and _live[0][0] is self:
            _free_engine()


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.fail("gpu-marked tests need a CUDA device (there is no CPU fallback to test)")
    assert torch.cuda.get_device_capability(0)[0] == 10, "kernels are sm_100a only"
    return torch.device("cuda:0")


@pytest.fixture(scope="module", params=SHAPE_IDS)
def case(request, dev):
    c = Case(SHAPES[request.param], dev)
    c.sid = request.param
    yield c
    c.close()


def rel_err(a, b):
    return ((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-12)).item()


RATIOS = {}   # (shape, layer): the largest err / bound of check A


@pytest.mark.gpu
def test_each_layer_alone_within_its_error_bound(case):
    """Check A: pbg_linear_bf16 of every layer on the reference's own bf16 operands, so that nothing differs but the
    accumulation.  Store layers: |got - ref| <= 1 bf16 ulp of |ref| + 2^-14 sum_k |a_k w_k|, padded columns exactly 0.
    D L1 logits: the accumulation term alone (through the LeakyReLU and w3).  G L2: 2e-3 (tanh.approx)."""
    ref, eng = case.ref, case.eng
    for B in batches(case.sid):
        xg, xd, _ = ref.inputs(case.node_emb, case.rel_w, *case.sample(B))
        g0, g1, gen, d0, logit = ref.forward(xg, xd)
        for name, (model, layer), a, want, lay in (("G L0", (0, 0), xg, g0, ref.g[0]), ("G L1", (0, 1), g0, g1, ref.g[1]),
                                                   ("D L0", (1, 0), xd, d0, ref.d[0])):
            got = eng.linear_bf16(model, layer, a.bfloat16().contiguous()).double()
            assert got.shape == want.shape
            assert bool((got[:, lay[2]:] == 0).all()), f"B = {B} {name}: padded columns are not 0"
            acc = ACC * (a.abs() @ lay[0].abs().T)
            r = ratio((got - want).abs(), ulp_bf16(want) + acc)
            RATIOS[(case.sid, name)] = max(RATIOS.get((case.sid, name), 0.0), r)
            assert r <= 1.0, f"B = {B} {name}: err / bound = {r:.3f}"
            # Where got != ref the two are neighbouring bf16 values (a rounding flip), and the exact activation lies at
            # least |y - midpoint| from the kernel's own fp32 value: the accumulation error the flip proves, over its term
            y = leaky(a @ lay[0].T + lay[1], ref.slope)
            flip = got != want
            r = ratio(torch.where(flip, (y - (got + want) / 2).abs(), 0.0), acc)
            RATIOS[(case.sid, name + " flips")] = max(RATIOS.get((case.sid, name + " flips"), 0.0), r)
        got = eng.linear_bf16(0, 2, g1.bfloat16().contiguous()).double()
        r = (got - gen).abs().max().item() / TANH_ATOL
        RATIOS[(case.sid, "G L2")] = max(RATIOS.get((case.sid, "G L2"), 0.0), r)
        assert r <= 1.0, f"B = {B} G L2: err / 2e-3 = {r:.3f}"
        got = eng.linear_bf16(1, 1, d0.bfloat16().contiguous()).double()
        r = ratio((got - logit).abs(), bound_rowdot(d0, ref.d[1][0], ref.d[1][1], ref.w3, ref.slope))
        RATIOS[(case.sid, "D L1")] = max(RATIOS.get((case.sid, "D L1"), 0.0), r)
        assert r <= 1.0, f"B = {B} D L1: err / bound = {r:.3f}"
    print(f"\ncheck A {case.sid} {case.dims}: largest err/bound " +
          ", ".join(f"{k[1]} {v:.3g}" for k, v in RATIOS.items() if k[0] == case.sid))
    eng.check_indices()


@pytest.mark.gpu
def test_fused_pass_equals_the_chain_of_single_layers(case):
    """Check B: the fused pass and the single-layer launches G0 -> G1 -> G2, D0 -> D1 use the same tiles, the same
    epilogue code and the same bias values (from shared or global memory), so they agree bit for bit."""
    ref, eng = case.ref, case.eng
    for B in batches(case.sid):
        trip, z = case.sample(B)
        xg, xd, t = ref.inputs(case.node_emb, case.rel_w, trip, z)
        c0 = eng.linear_bf16(0, 0, xg.bfloat16().contiguous())
        c1 = eng.linear_bf16(0, 1, c0)
        gen = eng.linear_bf16(0, 2, c1)
        logit = eng.linear_bf16(1, 1, eng.linear_bf16(1, 0, xd.bfloat16().contiguous()))
        f32 = case.run(trip, z)
        bf = case.run(trip, z, out_dtype=torch.bfloat16)
        assert torch.equal(f32["gen_out"], gen), f"B = {B}: gen_out (fp32) differs from the chain"
        assert torch.equal(bf["gen_out"], gen.bfloat16()), f"B = {B}: gen_out (bf16) differs from the chain"
        assert torch.equal(f32["logits"], logit) and torch.equal(bf["logits"], logit), f"B = {B}: logits differ"
        assert torch.equal(bf["gen_scores"], f32["gen_scores"]) and torch.equal(bf["probs"], f32["probs"])
        assert (f32["probs"].double() - torch.sigmoid(logit.double())).abs().max().item() <= 1e-6
        assert (f32["gen_scores"].double() - cosine64(gen, t)).abs().max().item() <= 1e-5
    eng.check_indices()


@pytest.mark.gpu
def test_fused_pass_against_the_float64_model(case):
    """Check C: the bf16 pass against the unrounded float64 model, at the project's bf16 bar (guards against an error the
    emulated reference shares with the kernels)."""
    for B in batches(case.sid):
        trip, z = case.sample(B)
        xg, xd, t = case.exact.inputs(case.node_emb, case.rel_w, trip, z)
        _, _, gen, _, logit = case.exact.forward(xg, xd)
        res = case.run(trip, z)
        assert rel_err(res["gen_out"], gen) <= 2e-2, f"B = {B}: gen_out"
        assert rel_err(res["logits"], logit) <= 2e-2, f"B = {B}: logits"
        assert rel_err(res["probs"], torch.sigmoid(logit)) <= 2e-2, f"B = {B}: probs"
        assert rel_err(res["gen_scores"], cosine64(gen, t)) <= 2e-2, f"B = {B}: gen_scores"
    case.eng.check_indices()


def check_fp32(res, exact, node_emb, rel_w, trip, z, gen=True, disc=True):
    """Check D: fp32 mode against the float64 model."""
    xg, xd, t = exact.inputs(node_emb, rel_w, trip, z)
    _, _, g, _, logit = exact.forward(xg, xd)
    if gen:
        assert (res["gen_out"].double() - g).abs().max().item() <= 1e-4
        assert (res["gen_scores"].double() - cosine64(g, t)).abs().max().item() <= 1e-4
    if disc:
        assert (res["probs"].double() - torch.sigmoid(logit)).abs().max().item() <= 1e-4
        assert (res["logits"].double() - logit).abs().max().item() <= 1e-4 * max(1.0, logit.abs().max().item())


@pytest.mark.gpu
def test_fp32_mode_against_the_float64_model(case):
    for B in batches(case.sid):
        trip, z = case.sample(B)
        check_fp32(case.run(trip, z, precision="fp32"), case.exact, case.node_emb, case.rel_w, trip, z)
    case.eng.check_indices()


def _equal(res, full, B, what):
    for k, v in res.items():
        assert torch.equal(v, full[k]), f"B = {B}, {what}: {k} differs from the full pass"


@pytest.mark.gpu
def test_generator_only_and_discriminator_only_passes(case):
    """Check E: at S4 / S8 these run another BIASS instance than the full pass."""
    for B in batches(case.sid):
        trip, z = case.sample(B)
        full = case.run(trip, z, out_dtype=torch.bfloat16)
        _equal(case.run(trip, z, out_dtype=torch.bfloat16, disc=False), full, B, "generator only")
        _equal(case.run(trip, z, gen=False), full, B, "discriminator only")
    case.eng.check_indices()


@pytest.mark.gpu
def test_staged_requests_on_both_slots(case):
    """Check E: stage_triplets (stage_rows_kernel) + score_staged = the fused pass, on both slots."""
    eng = case.eng
    for B in batches(case.sid):
        trip, z = case.sample(B)
        full = case.run(trip, z, out_dtype=torch.bfloat16)
        for slot in (0, 1):
            eng.stage_triplets(slot, case.node_emb, case.rel_w, trip, z)
            res = eng.score_staged(slot, want_gen_out=True, want_gen_scores=True, want_disc=True, out_dtype=torch.bfloat16)
            _equal(res, full, B, f"staged in slot {slot}")
    eng.check_indices()


@pytest.mark.gpu
def test_stage_next_chain_over_the_batches(case):
    """Check E: each pass gathers the next request into the other slot (the generic gather-ahead at every E != 128)."""
    eng = case.eng
    Bs = batches(case.sid)
    inputs = [case.sample(B) for B in Bs]
    full = [case.run(t, z, out_dtype=torch.bfloat16) for t, z in inputs]
    eng.reserve(max(Bs), "bf16", 2)
    eng.stage_triplets(0, case.node_emb, case.rel_w, *inputs[0])
    for j, B in enumerate(Bs):
        nxt = (case.node_emb, case.rel_w, *inputs[j + 1]) if j + 1 < len(Bs) else None
        res = eng.score_staged(j & 1, want_gen_out=True, want_gen_scores=True, want_disc=True, out_dtype=torch.bfloat16,
                               stage_next=nxt)
        _equal(res, full[j], B, "stage-next chain")
    eng.check_indices()


@pytest.mark.gpu
def test_two_cta_launch_width(case):
    eng = case.eng
    try:
        for B in batches(case.sid):
            trip, z = case.sample(B)
            full = case.run(trip, z, out_dtype=torch.bfloat16)
            eng.set_launch_width(2)
            res = case.run(trip, z, out_dtype=torch.bfloat16)
            eng.set_launch_width(0)
            _equal(res, full, B, "2 CTAs")
    finally:
        eng.set_launch_width(0)
    eng.check_indices()


@pytest.mark.gpu
def test_result_mirrors_with_guard_rows(case):
    """Check E: two mirrors with 64 guard rows behind the batch, bf16 and fp32 rows (bulk mirror stores when
    E % 64 == 0, per-lane stores otherwise); the guard rows must stay untouched."""
    eng, E, guard = case.eng, case.E, 64
    try:
        for B in batches(case.sid):
            trip, z = case.sample(B)
            for dt in (torch.bfloat16, torch.float32):
                full = case.run(trip, z, out_dtype=dt)
                mir = [{"gen_out": torch.full((B + guard, E), 7.0, dtype=dt, device=case.dev),
                        **{k: torch.full((B + guard,), 7.0, device=case.dev) for k in ("gen_scores", "logits", "probs")}}
                       for _ in range(2)]
                eng.set_result_mirrors(**{k: [d[k].data_ptr() for d in mir] for k in mir[0]})
                res = case.run(trip, z, out_dtype=dt)
                eng.set_result_mirrors()
                torch.cuda.synchronize()
                _equal(res, full, B, f"with mirrors ({dt})")
                for i, d in enumerate(mir):
                    for k, v in d.items():
                        assert torch.equal(v[:B], full[k]), f"B = {B} ({dt}): mirror {i} {k} differs"
                        assert bool((v[B:] == 7.0).all()), f"B = {B} ({dt}): mirror {i} {k}: guard rows were written"
    finally:
        eng.set_result_mirrors()
    eng.check_indices()


@pytest.mark.gpu
def test_trace_instance_gives_the_same_results(case):
    eng = case.eng
    try:
        for B in batches(case.sid):
            trip, z = case.sample(B)
            full = case.run(trip, z, out_dtype=torch.bfloat16)
            eng.debug_trace(True)
            res = case.run(trip, z, out_dtype=torch.bfloat16)
            trace = eng.debug_trace(False)
            _equal(res, full, B, "debug trace on")
            assert bool((trace != 0).any()), "the trace instance wrote no trace"
    finally:
        eng.debug_trace(False)
    eng.check_indices()


# --------------------------------------------------------------------------------------------- F: refusals and limits
@pytest.mark.gpu
@pytest.mark.parametrize("dims", [(12, 8, 64, 64, 0.2), (128, 64, 64, 24, 0.2), (128, 64, 64, 64, -0.1),
                                  (128, 64, 64, 64, 1.5)])
def test_create_refuses_unsupported_dims(dev, dims):
    from pbg import cabi
    with pytest.raises(cabi.PbgError) as ei:
        make_engine(dims, None, None, dev)
    assert ei.value.status == cabi.PBG_ERR_UNSUPPORTED


def _refused(fn):
    from pbg import cabi
    with pytest.raises(cabi.PbgError) as ei:
        fn()
    assert ei.value.status == cabi.PBG_ERR_UNSUPPORTED, str(ei.value)


@pytest.mark.gpu
@pytest.mark.parametrize("limit", ["embed_dim 520", "d_hidden 8208"])
def test_bf16_limits_are_refused_and_the_ctx_stays_usable(dev, limit):
    """embed_dim 520: a bf16 pass with the generator on is refused, a discriminator-only one passes check C.  d_hidden
    8208: a bf16 pass with the discriminator on is refused, a generator-only one passes check C.  fp32 mode passes
    check D at both, and after every refusal the same ctx runs a valid pass."""
    c = Case(LIMIT_E if limit == "embed_dim 520" else LIMIT_HD, dev)
    try:
        trip, z = c.sample(300)
        xg, xd, t = c.exact.inputs(c.node_emb, c.rel_w, trip, z)
        _, _, gen, _, logit = c.exact.forward(xg, xd)
        refused = [lambda: c.run(trip, z)]
        if limit == "embed_dim 520":
            refused.append(lambda: c.run(trip, z, disc=False))
        else:
            refused.append(lambda: c.run(trip, z, gen=False))
        for fn in refused:
            _refused(fn)
            if limit == "embed_dim 520":
                res = c.run(trip, z, gen=False)
                assert rel_err(res["logits"], logit) <= 2e-2 and rel_err(res["probs"], torch.sigmoid(logit)) <= 2e-2
            else:
                res = c.run(trip, z, disc=False)
                assert rel_err(res["gen_out"], gen) <= 2e-2 and rel_err(res["gen_scores"], cosine64(gen, t)) <= 2e-2
            check_fp32(c.run(trip, z, precision="fp32"), c.exact, c.node_emb, c.rel_w, trip, z)
        c.eng.check_indices()
    finally:
        c.close()
