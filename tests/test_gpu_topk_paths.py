"""Cosine top-k (pbg_topk) on every path it takes, judged by a float64 certificate.

``pbg_topk`` chooses between two pipelines and several branches inside each (csrc/pbg.cu: pbg_topk, topk_general):

  filter   E = 128, k <= 64, N >= max(4096, 64 stride k): bf16 sample scan (1 tile in ``stride``), cut-off per row,
           full scan into per-thread candidate lists, exact rescoring with a proof; a row that cannot be proven goes to
           the exact scan for one of four reasons (list overflow, too many candidates, too few, proof failed)
  general  everything else: exact fp32 scores of a chunk of rows (SIMT GEMM), then the histogram selection; a row with
           more than 2048 identical scores at the cut goes to the exact scan

``paths()`` restates those choices, and the case matrix below reaches every value.  Every answer is checked by
``certify()``, which needs no gap between scores: the returned scores must be the float64 cosines of the returned
indices, nothing left out may beat the k-th, and equal scores come back lower index first (include/pbg.h).

The tests without the gpu marker check the harness on the CPU: the certificate rejects each kind of wrong answer, the
branch map is reached, the selection kernel's fallback is reached, and the bf16 error bound holds where the old
constant did not.  Only one engine (one pbg_ctx) is alive at a time.
"""
import gc
import math
import re

import numpy as np
import pytest
import torch

# --------------------------------------------------------------------------------------------- the branch map
MAX_K_FILTER = 64        # kTkMaxK (topk_kernel.cuh)
SEL_BINS, SEL_CAP = 4096, 2048   # kSelBins, kSelCap


def sample_stride(k):
    return 4 if k <= 16 else 2          # tk_sample_stride


def paths(E, N, B, k):
    """The host's choices for one call, restated from csrc/pbg.cu (pbg_topk, topk_general, pbg_topk_prepare)."""
    stride = sample_stride(k)
    row_chunk = 4096 if k > 16 else 16384
    rows = [min(row_chunk, B - off) for off in range(0, B, row_chunk)]
    gen_rows = [max(64, min(r, (512 << 20) // (4 * N))) for r in rows]   # general path: rows per GEMM + selection
    return dict(
        filter=E == 128 and k <= MAX_K_FILTER and N >= max(16 * 256, 64 * stride * k),
        stride=stride, row_chunk=row_chunk, row_chunks=len(rows), last_rows=rows[-1],
        gen_chunks=sum(math.ceil(r / c) for r, c in zip(rows, gen_rows)),
        prepare="<8,1>" if E <= 128 else "<2,4>", reread=E > 512,
        tiles=(N + 255) // 256, last_tile_entities=N - (N + 255) // 256 * 256 + 256)


def select_flags_row(scores, k):
    """topk_select_kernel's decision for one row of fp32 scores, emulated in fp32 (tk_bin, tk_subbin, tk_find_bin):
    True when the row does not fit the kSelCap buffer and goes to topk_exact_kernel."""
    s = np.asarray(scores, dtype=np.float32)
    x = (s + np.float32(1.0)).astype(np.float32) * np.float32(SEL_BINS // 2)
    b = np.clip(x.astype(np.int64), 0, SEL_BINS - 1)                 # static_cast<int> truncates; x >= 0 here
    hist = np.bincount(b, minlength=SEL_BINS)

    def find(h, need):
        acc = 0
        for t in range(SEL_BINS - 1, -1, -1):
            if acc + h[t] >= need:
                return t, acc
            acc += h[t]
        raise AssertionError("fewer entries than k")
    T, above = find(hist, k)
    if above + hist[T] <= SEL_CAP:
        return False
    inT = b == T
    sub = np.clip(((x[inT] - np.float32(T)).astype(np.float32) * np.float32(SEL_BINS)).astype(np.int64), 0, SEL_BINS - 1)
    h2 = np.bincount(sub, minlength=SEL_BINS)
    T2, above2 = find(h2, k - above)
    return above + above2 + h2[T2] > SEL_CAP


# --------------------------------------------------------------------------------------------- the certificate
SCORE_TOL = 2e-6      # |returned score - float64 cosine of the returned index|
COMPLETE_TOL = 4e-6   # nothing left out may beat the k-th by more than this (fp32 evaluation noise, twice)


def normalized64(x):
    x = x.double()
    return x / x.norm(dim=1, keepdim=True).clamp_min(1e-12)


def certify(q, t, scores, idx, k, where=""):
    """Checks (scores, idx) = pbg_topk(q, t, k) row by row against S = normalize(q) @ normalize(t).T in float64,
    computed in row chunks on the inputs' device (B x N never more than 2^27 doubles at a time)."""
    B, N = q.shape[0], t.shape[0]
    assert scores.shape == (B, k) and idx.shape == (B, k) and idx.dtype == torch.int64, where
    dev = t.device
    tn = normalized64(t)
    scores, idx = scores.to(dev), idx.to(dev)
    step = max(1, (1 << 27) // N)
    for r0 in range(0, B, step):
        r1 = min(B, r0 + step)
        S = normalized64(q[r0:r1].to(dev)) @ tn.T
        sc, ix = scores[r0:r1], idx[r0:r1]
        rows = torch.arange(r0, r1, device=dev)
        bad = ((ix < 0) | (ix >= N)).any(dim=1)
        assert not bad.any(), f"{where}: index outside [0, N) in rows {rows[bad][:8].tolist()}"
        srt = ix.sort(dim=1).values
        dup = (srt[:, 1:] == srt[:, :-1]).any(dim=1) if k > 1 else torch.zeros_like(bad)
        assert not dup.any(), f"{where}: an index returned twice in rows {rows[dup][:8].tolist()}"
        sel = S.gather(1, ix)
        err = (sc.double() - sel).abs().amax(dim=1)
        assert (err <= SCORE_TOL).all(), f"{where}: score off its float64 cosine by {err.max().item():.3g}"
        if k > 1:
            inc = (sc[:, 1:] > sc[:, :-1]).any(dim=1)
            assert not inc.any(), f"{where}: scores not non-increasing in rows {rows[inc][:8].tolist()}"
            tie_order = ((sc[:, 1:] == sc[:, :-1]) & (ix[:, 1:] < ix[:, :-1])).any(dim=1)
            assert not tie_order.any(), f"{where}: equal scores not in ascending index order in rows {rows[tie_order][:8].tolist()}"
        kth = S.gather(1, ix[:, -1:])
        rest = S.scatter(1, ix, float("-inf"))
        over = rest.amax(dim=1, keepdim=True) - kth
        assert (over <= COMPLETE_TOL).all(), \
            f"{where}: an entity left out beats the k-th by {over.max().item():.3g} (row {r0 + int(over.argmax())})"
        # ties: a left-out entity whose float64 cosine EQUALS a returned one's must have the higher index
        lo = sel.amin(dim=1, keepdim=True)
        cand = (rest >= lo).nonzero()
        for c0 in range(0, cand.shape[0], 1 << 20):
            cr, cj = cand[c0:c0 + (1 << 20), 0], cand[c0:c0 + (1 << 20), 1]
            v = rest[cr, cj]
            beaten = ((sel[cr] == v[:, None]) & (ix[cr] > cj[:, None])).any(dim=1)
            assert not beaten.any(), (f"{where}: row {r0 + int(cr[beaten][0])} returns a higher index than the left-out "
                                      f"entity {int(cj[beaten][0])} of the same score")
        del S, rest


def ref_topk(q, t, k):
    """The certified answer in float64 (a stable sort: equal scores lower index first), scores as fp32."""
    S = normalized64(q) @ normalized64(t).T
    order = torch.sort(-S, dim=1, stable=True).indices[:, :k]
    return S.gather(1, order).float(), order


# --------------------------------------------------------------------------------------------- the bf16 error bound
OLD_ERR_BOUND = 0.0045
ERR_SLACK = 2e-5      # kTkErrSlack


def prepare_emulated(x):
    """topk_prepare_kernel's rounding on the CPU: fp32 normalisation, round to nearest even bf16.  Returns the
    normalised fp32 rows, their bf16 copies (as float64) and each row's rounding error ||bf16(x^) - x^|| (what
    topk_tau_kernel measures per query row and topk_prepare_kernel as a maximum over the table)."""
    x = x.float()
    inv = 1.0 / torch.clamp((x * x).sum(dim=1, keepdim=True).sqrt(), min=1e-12)
    xn = x * inv
    xb = xn.bfloat16().double()
    return xn, xb, (xb - xn.double()).norm(dim=1)


def err_bound(e_q, e_t):
    return e_q * (1 + e_t) + e_t + ERR_SLACK          # tk_err


DN = 2.0 ** -3 * (1 + 2.0 ** -8 - 2.0 ** -14)   # just below the midpoint 2^-3 (1 + 2^-8): rounds down by ~2^-8 relative
UP = 2.0 ** -3 * (1 + 2.0 ** -8 + 2.0 ** -14)   # just above it: rounds up by ~2^-8 relative


def unit_with(v, fix):
    v = v.clone()
    v[fix] = math.sqrt(1.0 - float((v * v).sum()))
    return v


def adversarial_needle_decoy(E=128, nA=33, nB=29, mA=0, beta=None):
    """A query q, a needle n and a decoy d (float64 unit vectors) such that the needle is the exact top-1 by less than
    0.002 while bf16 rounding pushes the needle's score down and the decoy's up: q and n share nA entries DN that
    round down; q and d share nB entries UP that round up, d has mA more UP entries on q's DN dimensions; d's entry
    beta on q's norm-fixing dimension tunes the margin."""
    q = torch.zeros(E, dtype=torch.float64)
    q[:nA] = DN
    q[nA:nA + nB] = UP
    q = unit_with(q, E - 2)
    n = torch.zeros(E, dtype=torch.float64)
    n[:nA] = DN
    n = unit_with(n, E - 3)

    def decoy(b):
        d = torch.zeros(E, dtype=torch.float64)
        d[:mA] = UP
        d[nA:nA + nB] = UP
        d[E - 2] = b
        return unit_with(d, E - 4)
    if beta is None:    # bisection: margin n.q - d.q = 0.001
        lo, hi = 0.0, 0.5
        for _ in range(60):
            mid = (lo + hi) / 2
            lo, hi = (lo, mid) if float(q @ decoy(mid)) > float(q @ n) - 0.001 else (mid, hi)
        beta = lo
    return q, n, decoy(beta)


# --------------------------------------------------------------------------------------------- CPU: the harness
def small_problem(seed=0, B=12, N=700, E=32):
    g = torch.Generator().manual_seed(seed)
    q, t = torch.randn(B, E, generator=g, dtype=torch.float64), torch.randn(N, E, generator=g, dtype=torch.float64)
    t[100:105] = 0.0                   # zero rows: exact ties at 0
    t[200] = t[201] = t[450] = q[0] * 3.0   # duplicates of the best row of query 0 (exact ties at 1.0)
    return q, t


def test_certificate_accepts_the_reference_answer_and_each_tie_break():
    q, t = small_problem()
    for k in (1, 3, 10, 40):
        s, i = ref_topk(q, t, k)
        certify(q, t, s, i, k, f"k={k}")
    s, i = ref_topk(q, t, 3)
    assert i[0].tolist() == [200, 201, 450]
    zq = torch.zeros(1, q.shape[1], dtype=torch.float64)
    s, i = ref_topk(zq, t, 5)
    assert i[0].tolist() == list(range(5))
    certify(zq, t, s, i, 5, "zero query")


def test_certificate_rejects_each_kind_of_wrong_answer():
    q, t = small_problem()
    k = 10
    s, i = ref_topk(q, t, k)
    s11, i11 = ref_topk(q, t, k + 1)
    S = normalized64(q) @ normalized64(t).T
    gap = S.gather(1, i11[:, k - 1:k]) - S.gather(1, i11[:, k:k + 1])
    r = int(gap.argmax())
    assert gap[r].item() > 1e-4
    swap_s, swap_i = s.clone(), i.clone()
    swap_i[r, -1] = i11[r, k]
    swap_s[r, -1] = s11[r, k]
    with pytest.raises(AssertionError, match="left out beats"):
        certify(q, t, swap_s, swap_i, k)
    neg = i.clone()
    neg[3, 4] = -1
    with pytest.raises(AssertionError, match="outside"):
        certify(q, t, s, neg, k)
    dup = i.clone()
    dup[3, 5] = dup[3, 4]
    with pytest.raises(AssertionError, match="twice"):
        certify(q, t, s, dup, k)
    off = s.clone()
    off[5, 2] += 1e-5
    with pytest.raises(AssertionError, match="off its float64"):
        certify(q, t, off, i, k)
    # ties: query 0's three best rows are duplicates 200, 201, 450
    hi_first = i.clone()
    hi_first[0, :2] = torch.tensor([201, 200])
    with pytest.raises(AssertionError, match="ascending index"):
        certify(q, t, s, hi_first, k)
    s2, i2 = ref_topk(q[:1], t, 2)
    with pytest.raises(AssertionError, match="higher index than the left-out"):   # 201, 450 instead of 200, 201
        certify(q[:1], t, s2, torch.tensor([[201, 450]]), 2)
    # the defect-1 form: zero rows 5 .. 9 returned where 0 .. 4 are due
    zq = torch.zeros(1, q.shape[1], dtype=torch.float64)
    zt = torch.cat([torch.zeros(20, q.shape[1], dtype=torch.float64), -t.abs()])
    zs, zi = ref_topk(zq, zt, 5)
    with pytest.raises(AssertionError, match="higher index than the left-out"):
        certify(zq, zt, zs, zi + 5, 5)


# --------------------------------------------------------------------------------------------- the case matrix
def needle_layout(num_sms, N, B, k):
    """Entities the needle sweep must use: N - 1, every tile's first and last entity, and the first and last entity of
    every tile at a boundary of a CTA pair's span in the scan and the sample launch (pbg.cu: pbg_topk, split)."""
    npairs = (num_sms & ~1) // 2
    rows_pad = (min(B, 4096 if k > 16 else 16384) + 255) // 256 * 256
    n_rb, n_tiles, stride = rows_pad // 256, (N + 255) // 256, sample_stride(k)
    must = {N - 1}
    for tiles, tstride, align in (((n_tiles + stride - 1) // stride, stride, True), (n_tiles, 1, False)):
        total = n_rb * tiles
        span = max(1, (total + npairs - 1) // npairs, (tiles + 14) // 15)
        if align and span < tiles:
            pieces = max(1, tiles // span)
            span = (tiles + pieces - 1) // pieces
        for u in range(0, total + 1, span):
            for v in (u - 1, u):
                if 0 <= v < total:
                    tile = (v % tiles) * tstride
                    must.update(e for e in (tile * 256, min(N, tile * 256 + 256) - 1) if e < N)
    return sorted(must)


# (name, E, N, B, k): the GPU cases whose paths the coverage test inspects
MATRIX = [
    ("filter k=1 N=4096", 128, 4096, 300, 1),
    ("general k=1 N=4095", 128, 4095, 300, 1),
    ("filter k=64 N=8192", 128, 8192, 300, 64),
    ("general k=64 N=8191", 128, 8191, 300, 64),
    ("filter two chunks, 1 row", 128, 8192, 16385, 16),
    ("filter k=17 ragged", 128, 4097, 4097, 17),
    ("general E=8", 8, 3000, 100, 10),
    ("general E=120", 120, 3000, 100, 10),
    ("general E=136", 136, 3000, 100, 10),
    ("general E=512", 512, 3000, 100, 10),
    ("general E=520", 520, 3000, 100, 10),
    ("general E=1024", 1024, 3000, 100, 10),
    ("general k=65", 128, 5000, 50, 65),
    ("general k=512", 128, 5000, 20, 512),
    ("general k=N=512", 128, 512, 10, 512),
    ("general 3 chunks", 64, 131072, 2500, 10),
]
NEEDLES = [(128, 65536 + 37, 4096, 16), (128, 65536 + 37, 4096, 64)]


def test_case_matrix_reaches_every_branch():
    p = [paths(E, N, B, k) for _, E, N, B, k in MATRIX + [(None, *c) for c in NEEDLES]]
    assert {x["filter"] for x in p} == {True, False}
    assert {x["stride"] for x in p if x["filter"]} == {2, 4}
    assert {x["row_chunk"] for x in p if x["filter"]} == {4096, 16384}
    assert any(x["filter"] and x["row_chunks"] > 1 and x["last_rows"] == 1 for x in p)
    assert any(x["filter"] and x["last_tile_entities"] == 1 for x in p)
    assert max(x["gen_chunks"] for x in p if not x["filter"]) == 3
    assert {(x["prepare"], x["reread"]) for x in p} == {("<8,1>", False), ("<2,4>", False), ("<2,4>", True)}
    # both sides of the path thresholds
    for (_, E, N, B, k), x in zip(MATRIX[:4], p[:4]):
        assert x["filter"] == (N == max(4096, 64 * sample_stride(k) * k))
    # the selection kernel's fallback: the tie case of test_tie_contract_general_path overflows kSelCap, a random row
    # and a crowded but distinct row do not
    tie = np.concatenate([np.full(3000, 0.3, np.float32), np.full(5, 0.9, np.float32), np.full(5192, -0.5, np.float32)])
    assert select_flags_row(tie, 10)
    rng = np.random.default_rng(0)
    assert not select_flags_row(rng.uniform(-0.4, 0.4, 8192).astype(np.float32), 10)
    assert not select_flags_row((0.3 + 1e-6 * np.arange(3000)).astype(np.float32), 10)


def test_old_constant_error_bound_is_exceeded_and_the_per_row_bound_holds():
    E = 128
    x = torch.zeros(E, dtype=torch.float64)
    x[:63] = DN * torch.where(torch.arange(63) % 2 == 0, 1.0, -1.0).double()
    x = unit_with(x, 100)
    xn, xb, e = prepare_emulated(x[None])
    exact = float(xn.double()[0] @ xn.double()[0])
    bf = float(xb[0] @ xb[0])
    assert abs(exact - 1.0) < 1e-6 and abs(bf - 0.99245) < 1e-4
    assert exact - bf > OLD_ERR_BOUND                       # the old constant was not a bound
    assert exact - bf <= err_bound(e[0].item(), e[0].item())
    # random rows: the per-row bound is no wider than the old constant
    g = torch.Generator().manual_seed(1)
    _, _, eq = prepare_emulated(torch.randn(4096, E, generator=g))
    _, _, et = prepare_emulated(torch.rand(65536, E, generator=g))
    assert err_bound(eq.max().item(), et.max().item()) < OLD_ERR_BOUND


def test_adversarial_needle_decoy_construction():
    q, n, d = adversarial_needle_decoy()
    xn, xb, e = prepare_emulated(torch.stack([q, n, d]))
    exact = xn.double() @ xn.double().T
    bf = xb @ xb.T
    margin = (exact[0, 1] - exact[0, 2]).item()
    e_needle, e_decoy = (exact[0, 1] - bf[0, 1]).item(), (bf[0, 2] - exact[0, 2]).item()
    assert 0 < margin < 0.002
    assert bf[0, 2] > bf[0, 1]                              # in bf16 the decoy wins
    assert e_needle + e_decoy > 0.0075, (e_needle, e_decoy)           # each close to 2^-8 ||q|| ||t||
    bound = err_bound(e[0].item(), e[1:].max().item())
    assert e_needle <= bound and e_decoy <= bound, (e_needle, e_decoy, bound)


# --------------------------------------------------------------------------------------------- GPU: one engine at a time
_live = []


def _free_engine():
    _live.clear()
    gc.collect()
    if torch.cuda.is_available():
        torch.cuda.synchronize()


def engine(E, dev):
    """Engine(E, 8, 8, 16, dev), reused while E stays the same; any other engine of this module is freed first."""
    from pbg.engine import Engine
    if _live and _live[0].E == E:
        return _live[0]
    _free_engine()
    eng = Engine(E, 8, 8, 16, dev)
    _live.append(eng)
    return eng


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.fail("gpu-marked tests need a CUDA device (there is no CPU fallback to test)")
    assert torch.cuda.get_device_capability(0)[0] == 10, "kernels are sm_100a only"
    yield torch.device("cuda:0")
    _free_engine()


REPORT = re.compile(r"(\d+) of (\d+) rows to the exact scan \(list overflow (\d+), too many candidates (\d+), "
                    r"too few (\d+), proof failed (\d+)\)")


def flag_counts(eng):
    """[flagged, overflow, too many, too few, proof failed] of the last chunk of the last call."""
    n = eng.topk_last_flagged()
    if n == 0:      # (after a general-path call the report is not rewritten)
        return [0, 0, 0, 0, 0]
    m = REPORT.search(eng.topk_flag_report)
    assert m, eng.topk_flag_report
    got = [int(m.group(1))] + [int(m.group(i)) for i in range(3, 7)]
    assert got[0] == n
    return got


def run(eng, q, t, k, where):
    s, i = eng.cosine_topk(q, t, k)
    certify(q, t, s, i, k, where)
    return s, i


def randn(g, *shape, dev):
    return torch.randn(*shape, generator=g).to(dev)


@pytest.mark.gpu
@pytest.mark.parametrize("case", MATRIX, ids=[c[0] for c in MATRIX])
def test_case_matrix(dev, case):
    name, E, N, B, k = case
    g = torch.Generator().manual_seed(MATRIX.index(case))
    eng = engine(E, dev)
    q, t = randn(g, B, E, dev=dev), randn(g, N, E, dev=dev)
    if k > 1:     # a few near-copies so that some rows have close scores near the top
        t[: min(N, 64)] = q[0] + 0.01 * randn(g, min(N, 64), E, dev=dev)
    run(eng, q, t, k, name)
    if paths(E, N, B, k)["filter"]:
        assert flag_counts(eng)[0] == 0, eng.topk_flag_report


@pytest.mark.gpu
def test_stale_state_between_calls(dev):
    """One engine through calls that change B, the table (same padded N, another tensor) and k: list slots, flags,
    cut-offs or candidate counts left over from an earlier call would show up as a wrong answer."""
    g = torch.Generator().manual_seed(3)
    eng = engine(128, dev)
    ta, tb = randn(g, 65536, 128, dev=dev), randn(g, 65436, 128, dev=dev)
    qa = randn(g, 16385, 128, dev=dev)
    for t, B, k in ((ta, 16385, 1), (ta, 1, 64), (tb, 4096, 10), (tb, 16385, 64), (ta, 1, 10), (tb, 300, 16)):
        run(eng, qa[:B], t, k, f"B={B} k={k} N={t.shape[0]}")
        assert flag_counts(eng)[0] == 0, eng.topk_flag_report


@pytest.mark.gpu
@pytest.mark.parametrize("E,N,k", [(128, 65536, 10), (128, 65536, 40), (64, 3000, 10)])
def test_row_norms_zero_rows_and_zero_query(dev, E, N, k):
    g = torch.Generator().manual_seed(N + k)
    eng = engine(E, dev)
    q = randn(g, 600, E, dev=dev)
    t = randn(g, N, E, dev=dev) * (10.0 ** (6 * torch.rand(N, 1, generator=g) - 3)).to(dev)
    q = q * (10.0 ** (6 * torch.rand(600, 1, generator=g) - 3)).to(dev)
    t[torch.randperm(N, generator=g)[:40].to(dev)] = 0.0
    q[7] = 0.0
    s, i = run(eng, q, t, k, f"E={E} N={N} k={k}")
    assert i[7].tolist() == list(range(k)), "a zero query ties every entity at 0: indices 0 .. k-1"
    assert (s[7] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("E,N,B,k", NEEDLES, ids=["k16-stride4", "k64-stride2"])
def test_needle_sweep_filter_path(dev, E, N, B, k):
    """Each planted row's k best entities are near-copies of its query (cosine ~ 0.99, the rest < 0.5), at positions
    that together cover every tile, both column halves, every group position and bit, entity N - 1 and the edges of
    every pair's span; the planted rows cover both CTA ranks, all epilogue warps and every lane."""
    assert paths(E, N, B, k)["filter"]
    g = torch.Generator().manual_seed(k)
    eng = engine(E, dev)
    q = randn(g, B, E, dev=dev)
    t = randn(g, N, E, dev=dev)
    n_rows = min(B, N // k)
    blocks = B // 256
    planted = torch.cat([torch.arange(b * 256, b * 256 + 256) for b in range(0, blocks, max(1, blocks * 256 // n_rows))])[:n_rows]
    assert set((planted % 256).tolist()) == set(range(256))
    must = needle_layout(torch.cuda.get_device_properties(0).multi_processor_count, N, B, k)
    rest = torch.randperm(N, generator=g)
    rest = rest[~torch.isin(rest, torch.tensor(must))]
    pos = torch.cat([torch.tensor(must), rest])[: planted.numel() * k].view(-1, k)
    used = pos.flatten()
    tiles, within = used // 256, used % 256
    assert set(tiles.tolist()) == set(range((N + 255) // 256)), "every tile"
    assert set((within // 128).tolist()) == {0, 1} and set(((within % 128) // 32).tolist()) == {0, 1, 2, 3}
    assert set((within % 32).tolist()) == set(range(32)) and N - 1 in used.tolist()
    noise = 0.14 * randn(g, planted.numel(), k, E, dev=dev)
    t[pos.to(dev)] = q[planted.to(dev)][:, None, :] + noise * q[planted.to(dev)].norm(dim=1)[:, None, None] / math.sqrt(E)
    s, i = run(eng, q, t, k, f"needles k={k}")
    assert (s[planted.to(dev)] > 0.95).all() and torch.equal(i[planted.to(dev)].sort(dim=1).values, pos.to(dev).sort(dim=1).values)
    assert flag_counts(eng)[0] == 0, eng.topk_flag_report


def band(g, q, n, lo, hi, dev):
    """n unit vectors whose cosines with the unit direction of q are spread over [lo, hi]."""
    E = q.numel()
    qh = q / q.norm()
    u = randn(g, n, E, dev=dev)
    u = u - (u @ qh)[:, None] * qh[None]
    u = u / u.norm(dim=1, keepdim=True)
    c = torch.linspace(lo, hi, n, device=dev)[torch.randperm(n, generator=g).to(dev)]
    return c[:, None] * qh[None] + (1 - c * c).sqrt()[:, None] * u


def orthogonal_to(q, x):
    """The rows of x with their component along q removed: a band around q then stays out of their cut-off."""
    qh = q / q.norm()
    return x - (x @ qh)[:, None] * qh[None]


@pytest.mark.gpu
def test_flag_reason_list_overflow(dev):
    """N = 262144 and B <= 256: a list covers 69 tiles (276 groups of 32 entities per column half); 4500 entities in the
    cut-off band of query 0, one in every 4 over the first span, overflow its list."""
    g = torch.Generator().manual_seed(41)
    eng = engine(128, dev)
    N, B, k = 262144, 64, 10
    t, q = randn(g, N, 128, dev=dev), randn(g, B, 128, dev=dev)
    q[1:] = orthogonal_to(q[0], q[1:])
    at = torch.arange(0, 18000, 4, device=dev)
    t[at] = band(g, q[0], at.numel(), 0.9985, 0.9995, dev)
    run(eng, q, t, k, "list overflow")
    got = flag_counts(eng)
    print("list overflow:", eng.topk_flag_report)
    assert got == [1, 1, 0, 0, 0], eng.topk_flag_report


@pytest.mark.gpu
def test_flag_reason_too_many_candidates(dev):
    """N = 65536, B = 4096: 2000 entities in query 0's cut-off band, one in each of 2000 groups spread over the table;
    no list can reach 256 groups (a pair's span is 56 tiles = 224 groups per half), the row has > 1024 candidates.
    The other queries are orthogonal to query 0, so that the band stays out of their cut-off."""
    g = torch.Generator().manual_seed(42)
    eng = engine(128, dev)
    N, B, k = 65536, 4096, 10
    t, q = randn(g, N, 128, dev=dev), randn(g, B, 128, dev=dev)
    q[1:] = orthogonal_to(q[0], q[1:])
    at = torch.arange(2000, device=dev) * 32 + 7
    t[at] = band(g, q[0], 2000, 0.9985, 0.9995, dev)
    run(eng, q, t, k, "too many candidates")
    got = flag_counts(eng)
    print("too many candidates:", eng.topk_flag_report)
    assert got == [1, 0, 1, 0, 0], eng.topk_flag_report


def defect1_table(E=128, N=65536, dev="cpu"):
    """Rows 0 .. 4999 zero, rows 5120 .. 5124 with cosines 0.50 .. 0.46 with e0, every other row about -e0.  Query
    e0 returns 5120 .. 5124 and then the zero rows 0 .. 4; query e0 - e1 has no positive cosine."""
    g = torch.Generator().manual_seed(7)
    t = torch.zeros(N, E)
    t[5000:, 0] = -1.0
    t[5000:, 2:] = 0.05 * torch.randn(N - 5000, E - 2, generator=g)
    for j in range(5):
        c = 0.5 - 0.01 * j
        t[5120 + j] = 0.0
        t[5120 + j, 0], t[5120 + j, 1] = c, math.sqrt(1 - c * c)
    q = torch.zeros(2, E)
    q[0, 0] = 1.0
    q[1, 0], q[1, 1] = 1.0, -1.0
    return q.to(dev), t.to(dev)


@pytest.mark.gpu
def test_flag_reason_too_few_candidates_and_tie_order(dev):
    """Five positive cosines for k = 10, so the row goes to the exact scan; there each thread t = 0 .. 4 holds zero rows
    t, t + 256, ... when row 5120 + t arrives, and must evict its highest-index zero row, not row t."""
    eng = engine(128, dev)
    q, t = defect1_table(dev=dev)
    assert paths(128, t.shape[0], 2, 10)["filter"]
    s, i = eng.cosine_topk(q, t, 10)
    got = flag_counts(eng)
    print("too few candidates:", eng.topk_flag_report, "row 0:", i[0].tolist())
    assert got == [2, 0, 0, 2, 0], eng.topk_flag_report
    assert i[0].tolist() == [5120, 5121, 5122, 5123, 5124, 0, 1, 2, 3, 4]
    assert i[1].tolist() == list(range(10))
    certify(q, t, s, i, 10, "too few candidates")


@pytest.mark.gpu
def test_flag_reason_proof_failed(dev):
    """No positive sampled key (tau = 0): 150 entities with cosines in (0.0005, 0.003), all in unsampled tiles, and
    every other entity at about -0.3.  The 10th exact score cannot beat tau by the error bound."""
    g = torch.Generator().manual_seed(44)
    eng = engine(128, dev)
    N, k = 65536, 10
    q = randn(g, 3, 128, dev=dev)
    t = band(g, q[0], N, -0.32, -0.28, dev)
    tiles = torch.arange(N // 256)
    unsampled = tiles[tiles % sample_stride(k) != 0]
    at = (unsampled[torch.randperm(unsampled.numel(), generator=g)[:150]] * 256
          + torch.randint(0, 256, (150,), generator=g)).to(dev)
    t[at] = band(g, q[0], 150, 0.0005, 0.003, dev)
    run(eng, q, t, k, "proof failed")
    got = flag_counts(eng)
    print("proof failed:", eng.topk_flag_report)
    assert got == [1, 0, 0, 0, 1], eng.topk_flag_report


@pytest.mark.gpu
@pytest.mark.parametrize("E,N,B,k", [(128, 65536, 512, 10), (128, 20000, 64, 80), (64, 20000, 64, 10)],
                         ids=["filter", "general-k80", "general-E64"])
def test_tie_contract_duplicate_best_rows(dev, E, N, B, k):
    """Each query's best row appears 12 times, at positions spread over tiles, column halves and list slots: the k
    lowest of those positions come back, in ascending order."""
    g = torch.Generator().manual_seed(N + k + E)
    eng = engine(E, dev)
    q, t = randn(g, B, E, dev=dev), randn(g, N, E, dev=dev)
    pos = torch.randperm(N, generator=g)[: B * 12].view(B, 12).to(dev)
    best = q + 0.05 * randn(g, B, E, dev=dev)
    t[pos] = best[:, None, :].expand(B, 12, E)
    s, i = run(eng, q, t, k, f"duplicates E={E} k={k}")
    want = pos.sort(dim=1).values[:, : min(k, 12)]
    assert torch.equal(i[:, : min(k, 12)], want)
    if paths(E, N, B, k)["filter"]:
        assert flag_counts(eng)[0] == 0, eng.topk_flag_report


@pytest.mark.gpu
def test_tie_contract_general_path_fallback(dev):
    """E = 64: 3000 identical rows at the cut (the selection kernel overflows kSelCap and flags the row) and better
    rows at 3072 + t, which land on exact-scan thread t next to its tied rows t, t + 256, ..."""
    E, N, k = 64, 8192, 10
    assert not paths(E, N, 1, k)["filter"]
    g = torch.Generator().manual_seed(5)
    eng = engine(E, dev)
    q = torch.zeros(1, E)
    q[0, 0] = 1.0
    t = torch.zeros(N, E)
    t[:, 0] = -1.0
    t[:, 2:] = 0.05 * torch.randn(N, E - 2, generator=g)
    t[:3000] = 0.0
    t[:3000, 0], t[:3000, 1] = 0.3, math.sqrt(1 - 0.09)
    for j in range(5):
        t[3072 + j] = 0.0
        t[3072 + j, 0], t[3072 + j, 1] = 0.9 - 0.01 * j, math.sqrt(1 - (0.9 - 0.01 * j) ** 2)
    sc = (normalized64(q) @ normalized64(t).T)[0].float().numpy()
    assert select_flags_row(sc, k)
    q, t = q.to(dev), t.to(dev)
    s, i = eng.cosine_topk(q, t, k)
    print("general fallback row 0:", i[0].tolist())
    assert i[0].tolist() == [3072, 3073, 3074, 3075, 3076, 0, 1, 2, 3, 4]
    certify(q, t, s, i, k, "general fallback")


@pytest.mark.gpu
def test_error_bound_adversarial_needle_and_decoys(dev):
    """The needle is the exact top-1 by < 0.002, but bf16 rounding lowers its score and raises 8 decoys' (in sampled
    tiles; the needle in an unsampled one).  The cut-off and the proof must account for the rounding error the
    prepare kernel measured."""
    qd, nd, dd = adversarial_needle_decoy()
    xn, xb, e = prepare_emulated(torch.stack([qd, nd, dd]))
    ex, bf = xn.double() @ xn.double().T, xb @ xb.T
    print(f"adversarial: margin {(ex[0, 1] - ex[0, 2]).item():.5f}, needle error {(ex[0, 1] - bf[0, 1]).item():.5f}, "
          f"decoy error {(bf[0, 2] - ex[0, 2]).item():.5f}, e_q {e[0].item():.5f}, e_t {e[1:].max().item():.5f}")
    g = torch.Generator().manual_seed(8)
    eng = engine(128, dev)
    N, k = 65536, 1
    q = torch.stack([qd.float()] + [torch.randn(128, generator=g) for _ in range(3)])
    t = band(g, qd.float(), N, -0.2, 0.2, "cpu")
    needle_at = 5 * 256 + 77                        # tile 5: not sampled at stride 4
    t[needle_at] = nd.float()
    decoys = torch.tensor([0, 4, 8, 40, 100, 128, 200, 252]) * 256 + 3   # sampled tiles
    t[decoys] = dd.float()
    q, t = q.to(dev), t.to(dev)
    s, i = run(eng, q, t, k, "adversarial bound")
    assert int(i[0, 0]) == needle_at
    assert flag_counts(eng)[0] == 0, eng.topk_flag_report
