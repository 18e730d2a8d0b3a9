"""Torch-tensor front end of the C ABI: one ``Engine`` = one ``pbg_ctx`` on one CUDA device.

PyTorch is plumbing here (device memory, streams); all arithmetic happens in libpbg_b200.so.
"""
from __future__ import annotations

import ctypes as C
import os

import torch
import torch.nn as nn

from . import cabi

_PRECISIONS = {"fp32": cabi.PREC_F32, "f32": cabi.PREC_F32, "float32": cabi.PREC_F32,
               "bf16": cabi.PREC_BF16, "bfloat16": cabi.PREC_BF16}


def default_precision() -> str:
    """``PBG_PRECISION`` env var (``bf16`` = tcgen05 fast mode, default; ``fp32`` = parity mode).

    An env var rather than a CLI flag so the reference's argparse surface stays untouched."""
    return os.environ.get("PBG_PRECISION", "bf16").lower()


def precision_code(precision: str | None) -> int:
    p = (precision or default_precision()).lower()
    if p not in _PRECISIONS:
        raise ValueError(f"unknown precision {p!r}; use 'fp32' or 'bf16'")
    return _PRECISIONS[p]


def fold_linear_bn(lin: nn.Linear, bn: nn.BatchNorm1d | None):
    """Fold an eval-mode BatchNorm1d into the preceding Linear (float64 arithmetic, fp32 result).

    Legal because the reference only runs the modules in eval mode under no_grad
    (pro_b_gan_infer.py:106-107, :133)."""
    W = lin.weight.detach().double().cpu()
    b = lin.bias.detach().double().cpu() if lin.bias is not None else torch.zeros(W.shape[0], dtype=torch.float64)
    if bn is not None:
        s = bn.weight.detach().double().cpu() / torch.sqrt(bn.running_var.detach().double().cpu() + bn.eps)
        W = W * s[:, None]
        b = (b - bn.running_mean.detach().double().cpu()) * s + bn.bias.detach().double().cpu()
    return W.float().contiguous(), b.float().contiguous()


def _ptr(t: torch.Tensor | None):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class Engine:
    """Owns a pbg_ctx.  Methods take / return CUDA tensors on the engine's device."""

    def __init__(self, embed_dim: int, noise_dim: int, g_hidden: int, d_hidden: int,
                 device: torch.device | str | int, leaky_slope: float = 0.2, ctas: int = 0):
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError(f"pro-b-gan_b200 runs only on CUDA (sm_100a) devices, got {device}; there is no CPU fallback")
        if not torch.cuda.is_available():
            raise RuntimeError("pro-b-gan_b200: no CUDA device is available and there is no CPU fallback")
        self.device = torch.device("cuda", device.index if device.index is not None else torch.cuda.current_device())
        self.E, self.Z, self.HG, self.HD = int(embed_dim), int(noise_dim), int(g_hidden), int(d_hidden)
        self._lib = cabi.load()
        self._h = C.c_void_p(0)
        dims = cabi.PbgDims(self.E, self.Z, self.HG, self.HD, self.device.index, float(leaky_slope))
        st = self._lib.pbg_create(C.byref(self._h), C.byref(dims))
        if st != cabi.PBG_OK:
            self._h = C.c_void_p(0)
            cabi.check(st, None)
        self.g_loaded = self.d_loaded = False
        self._latent_on = False
        if ctas:
            self.set_launch_width(ctas)

    def set_launch_width(self, ctas: int) -> None:
        """CTAs (SMs) one fused pass occupies; 0 = the whole device.  See include/pbg.h."""
        cabi.check(self._lib.pbg_set_launch_width(self._h, int(ctas)), self._h)

    def last_pass_sm_clock(self) -> float:
        """SM clock (MHz) during this ctx's last bf16-mode pass, measured in the kernel (include/pbg.h); synchronises."""
        import ctypes
        mhz = ctypes.c_double(0.0)
        with torch.cuda.device(self.device):
            cabi.check(self._lib.pbg_last_pass_sm_clock(self._h, self._stream(), ctypes.byref(mhz)), self._h)
        return float(mhz.value)

    def set_workspace_discard(self, on: bool) -> None:
        """Dead activation row blocks are dropped from L2 instead of being written back to HBM (default on).  See include/pbg.h."""
        cabi.check(self._lib.pbg_set_workspace_discard(self._h, int(bool(on))), self._h)

    def cosine_topk(self, queries: torch.Tensor, table: torch.Tensor, k: int):
        """``F.normalize(queries) @ F.normalize(table).T`` followed by ``.topk(k, dim=1)`` without the [B, N] matrix
        (pro_b_gan_infer.py:146-151, :231-236).  Returns (scores fp32 [B, k], indices int64 [B, k]) like torch.topk.
        The prepared (normalised) table is cached until the tensor is modified or another table is passed."""
        table = self._f32(table, self.E, "table")
        queries = self._f32(queries, self.E, "queries")
        self.validate_top_k(k, table.shape[0])
        key = (table.data_ptr(), tuple(table.shape), table._version)
        with torch.cuda.device(self.device):
            if getattr(self, "_topk_key", None) != key:
                cabi.check(self._lib.pbg_topk_prepare(self._h, _ptr(table), table.shape[0], self._stream()), self._h)
                self._topk_key, self._topk_table = key, table   # keep the tensor alive while the ctx refers to it
            B = queries.shape[0]
            scores = torch.empty(B, k, dtype=torch.float32, device=self.device)
            idx = torch.empty(B, k, dtype=torch.int64, device=self.device)
            cabi.check(self._lib.pbg_topk(self._h, _ptr(queries), B, int(k), _ptr(idx), _ptr(scores), self._stream()), self._h)
        return scores, idx

    def topk_last_flagged(self) -> int:
        """Rows of the last cosine_topk call (its last 16384-row chunk) that went to the exact scan; synchronises."""
        n = int(self._lib.pbg_topk_last_flagged(self._h, self._stream()))
        self.topk_flag_report = cabi.last_error(self._h)    # "… rows to the exact scan (list overflow a, …, proof failed d)"
        return n

    MAX_TOP_K = 512   # include/pbg.h: pbg_topk selects up to 512 per row on the device

    @classmethod
    def validate_top_k(cls, k: int, num_rows: int) -> None:
        """The errors of ``similarities.topk(k, dim=1)`` (pro_b_gan_infer.py:151, :236) plus this library's own limit,
        raised on the host before anything is launched."""
        if k > num_rows:
            raise RuntimeError(f"selected index k out of range: k = {k} > {num_rows} rows")  # what torch.topk raises
        if k < 1:
            raise RuntimeError(f"top_k must be positive, got {k}")
        if k > cls.MAX_TOP_K:
            raise NotImplementedError(f"top_k = {k}: the CUDA path selects at most {cls.MAX_TOP_K} per row "
                                      "(k <= 64 on the tensor-core filter, above that exact fp32 scores + selection)")

    def set_result_mirrors(self, gen_out=(), gen_scores=(), logits=(), probs=()) -> None:
        """Device addresses (ints) of up to 7 mirror buffers per result, e.g. peer GPUs' windows: every bf16-mode
        pass also writes its rows there (include/pbg.h: pbg_set_result_mirrors).  Empty lists clear."""
        n = max(len(gen_out), len(gen_scores), len(logits), len(probs))
        def arr(ptrs):
            if not ptrs:
                return None
            if len(ptrs) != n:
                raise ValueError("every given mirror list must have the same length")
            return (C.c_void_p * n)(*[C.c_void_p(int(x)) for x in ptrs])
        a = [arr(gen_out), arr(gen_scores), arr(logits), arr(probs)]
        cabi.check(self._lib.pbg_set_result_mirrors(self._h, n, *[C.cast(x, C.c_void_p) if x is not None else None for x in a]),
                   self._h)

    def set_result_multicast(self, gen_out: int = 0, gen_scores: int = 0, logits: int = 0, probs: int = 0) -> None:
        """NVSwitch multicast addresses (ints) of symmetric result buffers, offset to this rank's shard: every bf16-mode
        pass also writes its rows there with multimem.st (include/pbg.h: pbg_set_result_multicast).  All 0 clears."""
        cabi.check(self._lib.pbg_set_result_multicast(self._h, *[C.c_void_p(int(x)) if x else None
                                                                 for x in (gen_out, gen_scores, logits, probs)]), self._h)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            try:
                self._lib.pbg_destroy(h)
            except Exception:
                pass
            self._h = C.c_void_p(0)

    # ------------------------------------------------------------------ weights
    def load_generator(self, layers) -> None:
        """layers: [(W1,b1),(W2,b2),(W3,b3)] fp32 CPU tensors, BatchNorm already folded."""
        blob = torch.cat([t.reshape(-1).float().cpu() for wb in layers for t in wb]).contiguous()
        cabi.check(self._lib.pbg_load_generator(self._h, C.c_void_p(blob.data_ptr()), blob.numel()), self._h)
        self.g_loaded = True

    def load_discriminator(self, layers) -> None:
        """layers: [(W1,b1),(W2,b2),(w3,b3)] fp32 CPU tensors."""
        blob = torch.cat([t.reshape(-1).float().cpu() for wb in layers for t in wb]).contiguous()
        cabi.check(self._lib.pbg_load_discriminator(self._h, C.c_void_p(blob.data_ptr()), blob.numel()), self._h)
        self.d_loaded = True

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _f32(self, t: torch.Tensor, cols: int, name: str) -> torch.Tensor:
        if t.device != self.device:
            raise RuntimeError(f"{name} is on {t.device}, engine is on {self.device}")
        if t.dim() != 2 or t.shape[1] != cols:
            raise ValueError(f"{name} must be [B, {cols}], got {tuple(t.shape)}")
        return t.detach().to(torch.float32).contiguous()

    def _i64(self, t: torch.Tensor, name: str) -> torch.Tensor:
        if t.device != self.device:
            raise RuntimeError(f"{name} is on {t.device}, engine is on {self.device}")
        return t.detach().to(torch.int64)

    def check_indices(self) -> None:
        """Synchronise and raise IndexError if a gather since the last check saw an out-of-range id."""
        cabi.check(self._lib.pbg_check_indices(self._h, self._stream()), self._h)

    def profile_enable(self, on: bool = True) -> None:
        cabi.check(self._lib.pbg_profile_enable(self._h, 1 if on else 0), self._h)

    def profile_read(self) -> dict:
        """{kind: (total_ms, launches)} since the last read; synchronises the device."""
        n = len(cabi.KERNEL_KINDS)
        ms = (C.c_double * n)(*([0.0] * n))
        cnt = (C.c_int64 * n)(*([0] * n))
        cabi.check(self._lib.pbg_profile_read(self._h, ms, cnt), self._h)
        return {k: (ms[i], cnt[i]) for i, k in enumerate(cabi.KERNEL_KINDS)}

    def debug_trace(self, enable: bool = True):
        """Read the per-CTA clock64 trace slots ([num_SMs, 256] int64 tensor), then enable / disable tracing and
        zero the buffer."""
        n = torch.cuda.get_device_properties(self.device).multi_processor_count * 256
        buf = (C.c_int64 * n)()
        cabi.check(self._lib.pbg_debug_trace(self._h, 1 if enable else 0, buf, n), self._h)
        return torch.tensor(list(buf), dtype=torch.int64).reshape(-1, 256)

    @property
    def launch_count(self) -> int:
        return int(self._lib.pbg_launch_count(self._h))

    # ------------------------------------------------------------------ device latents
    def set_latent_stream(self, enable: bool = True, seed: int = 0, offset: int = 0) -> None:
        """Turn the ctx's latent stream on or off (include/pbg.h: pbg_set_latent_stream).  While it is on, every generator
        call given ``z=None`` draws its [B, Z] latents on the device exactly as ``torch.randn((B, Z), device=...,
        generator=g)`` would for a CUDA generator at Philox (seed, offset), and advances the offset the same way.
        Synchronises the device."""
        with torch.cuda.device(self.device):
            cabi.check(self._lib.pbg_set_latent_stream(self._h, int(bool(enable)), int(seed), int(offset)), self._h)
        self._latent_on = bool(enable)

    def latent_stream(self) -> tuple[int, int]:
        """(seed, offset) of the ctx's latent stream: where the next draw starts.  Synchronises the current stream."""
        seed, off = C.c_uint64(0), C.c_uint64(0)
        with torch.cuda.device(self.device):
            cabi.check(self._lib.pbg_get_latent_stream(self._h, C.byref(seed), C.byref(off), self._stream()), self._h)
        return int(seed.value), int(off.value)

    def draw_latents(self, rows: int, seed: int, offset: int, row_begin: int = 0,
                     total_rows: int | None = None) -> tuple[torch.Tensor, int]:
        """Rows [row_begin, row_begin + rows) of the draw ``torch.randn((total_rows, Z), device=..., generator=g)`` makes
        for g at Philox (seed, offset) (total_rows defaults to rows), as a new fp32 [rows, Z] tensor; with the offset the
        generator has after that draw.  Stateless: the ctx's own stream does not move."""
        total = int(rows if total_rows is None else total_rows)
        z = torch.empty(int(rows), self.Z, dtype=torch.float32, device=self.device)
        after = C.c_uint64(0)
        with torch.cuda.device(self.device):
            cabi.check(self._lib.pbg_draw_latents(self._h, int(seed), int(offset), total, int(row_begin), int(rows), _ptr(z),
                                                  C.byref(after), self._stream()), self._h)
        return z, int(after.value)

    def _latents(self, z, name: str = "z"):
        """The caller's latents, or None (drawn by the ctx) when the latent stream is on."""
        if z is not None:
            return self._f32(z, self.Z, name)
        if not self._latent_on:
            raise ValueError("generator pass needs latents z (or the ctx's latent stream: set_latent_stream)")
        return None

    # ------------------------------------------------------------------ generator
    def generator_forward(self, h, r, z=None, precision=None, out_dtype=torch.float32) -> torch.Tensor:
        h, r, z = self._f32(h, self.E, "h_emb"), self._f32(r, self.E, "r_emb"), self._latents(z)
        B = h.shape[0]
        if r.shape[0] != B or (z is not None and z.shape[0] != B):
            raise ValueError("h_emb, r_emb and z must have the same batch size")
        out = torch.empty(B, self.E, dtype=out_dtype, device=self.device)
        with torch.cuda.device(self.device):
            cabi.check(self._lib.pbg_generator_forward(
                self._h, _ptr(h), _ptr(r), _ptr(z), _ptr(out), B, precision_code(precision),
                cabi.DT_BF16 if out_dtype == torch.bfloat16 else cabi.DT_F32, self._stream()), self._h)
        return out

    def generator_forward_gather(self, node_emb, rel_w, heads, rels, z=None, precision=None,
                                 out_dtype=torch.float32) -> torch.Tensor:
        node_emb = self._f32(node_emb, self.E, "node_emb")
        rel_w = self._f32(rel_w, self.E, "rel_emb.weight")
        heads, rels = self._i64(heads, "heads"), self._i64(rels, "relations")
        z = self._latents(z)
        B = heads.shape[0]
        out = torch.empty(B, self.E, dtype=out_dtype, device=self.device)
        with torch.cuda.device(self.device):
            cabi.check(self._lib.pbg_generator_forward_gather(
                self._h, _ptr(node_emb), node_emb.shape[0], _ptr(rel_w), rel_w.shape[0],
                _ptr(heads), heads.stride(0) if B else 1, _ptr(rels), rels.stride(0) if B else 1, _ptr(z), _ptr(out),
                B, precision_code(precision), cabi.DT_BF16 if out_dtype == torch.bfloat16 else cabi.DT_F32,
                self._stream()), self._h)
        return out

    # ------------------------------------------------------------------ discriminator
    def discriminator_forward(self, h, r, t, precision=None):
        h, r, t = self._f32(h, self.E, "h_emb"), self._f32(r, self.E, "r_emb"), self._f32(t, self.E, "t_emb")
        B = h.shape[0]
        logits = torch.empty(B, dtype=torch.float32, device=self.device)
        probs = torch.empty(B, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            cabi.check(self._lib.pbg_discriminator_forward(
                self._h, _ptr(h), _ptr(r), _ptr(t), _ptr(logits), _ptr(probs), B, precision_code(precision),
                self._stream()), self._h)
        return logits, probs

    def linear_bf16(self, model: int, layer: int, a_bf16: torch.Tensor) -> torch.Tensor:
        """Per-layer diagnostic: one tensor-core Linear (+ its fused epilogue) on a bf16 [M, Kp] matrix."""
        if a_bf16.dtype != torch.bfloat16 or a_bf16.device != self.device or not a_bf16.is_contiguous():
            raise ValueError("a_bf16 must be a contiguous bf16 tensor on the engine's device")
        M = a_bf16.shape[0]
        if model == 0 and layer == 2:
            out = torch.empty(M, self.E, dtype=torch.float32, device=self.device)
        elif model == 1 and layer == 1:
            out = torch.empty(M, dtype=torch.float32, device=self.device)
        else:
            width = (self.HG if model == 0 else self.HD)
            out = torch.empty(M, (width + 127) // 128 * 128, dtype=torch.bfloat16, device=self.device)
        with torch.cuda.device(self.device):
            cabi.check(self._lib.pbg_linear_bf16(self._h, model, layer, _ptr(a_bf16), _ptr(out), M, self._stream()),
                       self._h)
        return out

    # ------------------------------------------------------------------ fused G + D pass
    def score_triplets(self, node_emb, rel_w, triplets, z=None, want_gen_out=False, want_gen_scores=False,
                       want_disc=True, precision=None, out_dtype=torch.float32, out: dict | None = None):
        """One gather feeding G and/or D.  Returns dict with the requested tensors.

        ``out`` may carry preallocated result tensors (keys gen_out / gen_scores / logits / probs) so that a
        steady-state caller (bench.py, CUDA-graph capture) performs no allocation per call."""
        node_emb = self._f32(node_emb, self.E, "node_emb")
        rel_w = self._f32(rel_w, self.E, "rel_emb.weight")
        trip = self._i64(triplets, "triplets")
        if trip.dim() != 2 or trip.shape[1] != 3:
            raise ValueError(f"triplets must be [B, 3], got {tuple(trip.shape)}")
        trip = trip.contiguous()
        B = trip.shape[0]
        run_g = want_gen_out or want_gen_scores
        if run_g:
            z = self._latents(z)
        res = {}
        out = out or {}

        def buf(key, want, shape, dtype):
            if not want:
                return None
            t = out.get(key)
            if t is None:
                return torch.empty(shape, dtype=dtype, device=self.device)
            if tuple(t.shape) != tuple(shape) or t.dtype != dtype or t.device != self.device or not t.is_contiguous():
                raise ValueError(f"out[{key!r}] must be a contiguous {dtype} tensor of shape {tuple(shape)} on {self.device}")
            return t

        gen_out = buf("gen_out", want_gen_out, (B, self.E), out_dtype)
        scores = buf("gen_scores", want_gen_scores, (B,), torch.float32)
        logits = buf("logits", want_disc, (B,), torch.float32)
        probs = buf("probs", want_disc, (B,), torch.float32)
        with torch.cuda.device(self.device):
            cabi.check(self._lib.pbg_score_triplets(
                self._h, _ptr(node_emb), node_emb.shape[0], _ptr(rel_w), rel_w.shape[0], _ptr(trip),
                _ptr(z if run_g else None), _ptr(gen_out),
                cabi.DT_BF16 if out_dtype == torch.bfloat16 else cabi.DT_F32,
                _ptr(scores), _ptr(logits), _ptr(probs), B, precision_code(precision), self._stream()), self._h)
        if want_gen_out:
            res["gen_out"] = gen_out
        if want_gen_scores:
            res["gen_scores"] = scores
        if want_disc:
            res["logits"], res["probs"] = logits, probs
        return res

    # ------------------------------------------------------------------ staged requests (ingest / compute split)
    def reserve(self, rows: int, precision=None, stage_slots: int = 0) -> None:
        """Size the workspaces (and staging slots) for `rows` rows up front (include/pbg.h: pbg_reserve): nothing then
        grows -- no device synchronisation -- inside a steady-state loop or a CUDA-graph capture."""
        with torch.cuda.device(self.device):
            cabi.check(self._lib.pbg_reserve(self._h, int(rows), precision_code(precision), int(stage_slots)), self._h)

    def stage_triplets(self, slot: int, node_emb, rel_w, triplets, z=None, want_gen=True, want_disc=True) -> int:
        """Gather + concat + cast one request's rows into staging slot `slot` on the CURRENT stream (the caller's ingest
        stream), beside whatever pass is running.  Returns the request's row count.  See pbg_stage_triplets."""
        node_emb = self._f32(node_emb, self.E, "node_emb")
        rel_w = self._f32(rel_w, self.E, "rel_emb.weight")
        trip = self._i64(triplets, "triplets")
        if trip.dim() != 2 or trip.shape[1] != 3:
            raise ValueError(f"triplets must be [B, 3], got {tuple(trip.shape)}")
        trip = trip.contiguous()
        if want_gen:
            z = self._latents(z)
        B = trip.shape[0]
        with torch.cuda.device(self.device):
            cabi.check(self._lib.pbg_stage_triplets(
                self._h, int(slot), _ptr(node_emb), node_emb.shape[0], _ptr(rel_w), rel_w.shape[0], _ptr(trip),
                _ptr(z if want_gen else None), B, 1 if want_gen else 0, 1 if want_disc else 0, self._stream()), self._h)
        if not hasattr(self, "_staged_rows"):
            self._staged_rows = {}
        self._staged_rows[int(slot)] = B
        return B

    def score_staged(self, slot: int, want_gen_out=False, want_gen_scores=False, want_disc=True,
                     out_dtype=torch.float32, out: dict | None = None, stage_next: tuple | None = None):
        """The G + D pass over a staged request on the CURRENT stream (the compute stream); the caller has ordered it
        after the slot's stage_triplets.  Same result dict as score_triplets (bf16 mode).
        ``stage_next = (node_emb, rel_w, triplets, z)``: the same launch also stages that request into the other slot
        (pbg_score_staged_stage_next) -- its tensors must stay alive until it has been scored -- and CONSUMES `slot`:
        stage it again before scoring it again."""
        res, out = {}, (out or {})
        B = getattr(self, "_staged_rows", {}).get(int(slot))
        if B is None:
            raise ValueError(f"nothing staged in slot {slot}")

        def buf(key, want, shape, dtype):
            if not want:
                return None
            t = out.get(key)
            if t is None:
                return torch.empty(shape, dtype=dtype, device=self.device)
            if tuple(t.shape) != tuple(shape) or t.dtype != dtype or t.device != self.device or not t.is_contiguous():
                raise ValueError(f"out[{key!r}] must be a contiguous {dtype} tensor of shape {tuple(shape)} on {self.device}")
            return t

        gen_out = buf("gen_out", want_gen_out, (B, self.E), out_dtype)
        scores = buf("gen_scores", want_gen_scores, (B,), torch.float32)
        logits = buf("logits", want_disc, (B,), torch.float32)
        probs = buf("probs", want_disc, (B,), torch.float32)
        dt = cabi.DT_BF16 if out_dtype == torch.bfloat16 else cabi.DT_F32
        with torch.cuda.device(self.device):
            if stage_next is None:
                cabi.check(self._lib.pbg_score_staged(self._h, int(slot), _ptr(gen_out), dt, _ptr(scores), _ptr(logits),
                                                      _ptr(probs), self._stream()), self._h)
            else:
                n_emb, n_rel, n_trip, n_z = stage_next
                n_emb, n_rel = self._f32(n_emb, self.E, "node_emb"), self._f32(n_rel, self.E, "rel_emb.weight")
                n_trip = self._i64(n_trip, "triplets")
                if n_trip.dim() != 2 or n_trip.shape[1] != 3 or not n_trip.is_contiguous():
                    raise ValueError("the next request's triplets must be a contiguous [B, 3] tensor")
                run_g = want_gen_out or want_gen_scores
                if run_g:
                    n_z = self._latents(n_z)
                cabi.check(self._lib.pbg_score_staged_stage_next(
                    self._h, int(slot), _ptr(gen_out), dt, _ptr(scores), _ptr(logits), _ptr(probs), _ptr(n_emb), n_emb.shape[0],
                    _ptr(n_rel), n_rel.shape[0], _ptr(n_trip), _ptr(n_z if run_g else None), n_trip.shape[0], self._stream()),
                    self._h)
                self._staged_rows.pop(int(slot), None)            # consumed by this call (include/pbg.h)
                self._staged_rows[1 - int(slot)] = n_trip.shape[0]
                if not hasattr(self, "_staged_keep"):
                    self._staged_keep = {}
                self._staged_keep[1 - int(slot)] = (n_emb, n_rel, n_trip, n_z)   # alive until that slot is staged again
        if want_gen_out:
            res["gen_out"] = gen_out
        if want_gen_scores:
            res["gen_scores"] = scores
        if want_disc:
            res["logits"], res["probs"] = logits, probs
        return res

    def score_triplets_host(self, node_emb, rel_w, triplets_host, z_host=None, gen_out_host=None,
                            gen_scores_host=None, logits_host=None, probs_host=None, precision=None) -> None:
        """End-to-end form: index / latent / result buffers are HOST tensors (ideally pinned); the H2D and
        D2H copies happen inside the call, which returns after one stream synchronise."""
        for name, t in (("triplets", triplets_host), ("z", z_host), ("gen_out", gen_out_host),
                        ("gen_scores", gen_scores_host), ("logits", logits_host), ("probs", probs_host)):
            if t is not None and (t.device.type != "cpu" or not t.is_contiguous()):
                raise ValueError(f"{name}_host must be a contiguous CPU tensor")
        if triplets_host.dtype != torch.int64 or triplets_host.dim() != 2 or triplets_host.shape[1] != 3:
            raise ValueError("triplets_host must be int64 [B, 3]")
        B = triplets_host.shape[0]
        with torch.cuda.device(self.device):
            cabi.check(self._lib.pbg_score_triplets_host(
                self._h, _ptr(node_emb), node_emb.shape[0], _ptr(rel_w), rel_w.shape[0], _ptr(triplets_host),
                _ptr(z_host), _ptr(gen_out_host), _ptr(gen_scores_host), _ptr(logits_host), _ptr(probs_host),
                B, precision_code(precision)), self._h)

    def score_triplets_host_packed(self, node_emb, rel_w, in_block_host: torch.Tensor, out_block_host: torch.Tensor,
                                   B: int, precision=None) -> None:
        """pbg_score_triplets_host_packed: ``in_block_host`` = uint8 [24 B + 4 Z B] holding [triplets int64 | z fp32],
        ``out_block_host`` = fp32 [3 B] receiving [gen_scores | logits | probs]; one copy per direction, one sync."""
        if in_block_host.device.type != "cpu" or out_block_host.device.type != "cpu":
            raise ValueError("the blocks must be CPU (ideally pinned) tensors")
        if in_block_host.numel() * in_block_host.element_size() != B * (24 + 4 * self.Z) or not in_block_host.is_contiguous():
            raise ValueError(f"in_block_host must hold {B * (24 + 4 * self.Z)} contiguous bytes")
        if out_block_host.dtype != torch.float32 or out_block_host.numel() != 3 * B or not out_block_host.is_contiguous():
            raise ValueError(f"out_block_host must be a contiguous fp32 tensor of {3 * B} elements")
        with torch.cuda.device(self.device):
            cabi.check(self._lib.pbg_score_triplets_host_packed(
                self._h, _ptr(node_emb), node_emb.shape[0], _ptr(rel_w), rel_w.shape[0], _ptr(in_block_host),
                _ptr(out_block_host), B, precision_code(precision)), self._h)

    def score_triplets_host_ids(self, node_emb, rel_w, triplets_host: torch.Tensor, out_block_host: torch.Tensor,
                                precision=None) -> None:
        """pbg_score_triplets_host_ids: only the ids travel -- ``triplets_host`` int64 [B, 3] in, ``out_block_host`` fp32
        [3 B] = [gen_scores | logits | probs] out -- and the latents come from the ctx's latent stream, which must be on.
        One copy per direction, one sync."""
        if triplets_host.device.type != "cpu" or out_block_host.device.type != "cpu":
            raise ValueError("the blocks must be CPU (ideally pinned) tensors")
        if triplets_host.dtype != torch.int64 or triplets_host.dim() != 2 or triplets_host.shape[1] != 3 \
                or not triplets_host.is_contiguous():
            raise ValueError("triplets_host must be a contiguous int64 [B, 3] tensor")
        B = triplets_host.shape[0]
        if out_block_host.dtype != torch.float32 or out_block_host.numel() != 3 * B or not out_block_host.is_contiguous():
            raise ValueError(f"out_block_host must be a contiguous fp32 tensor of {3 * B} elements")
        if not self._latent_on:
            raise ValueError("score_triplets_host_ids draws the latents on the device: call set_latent_stream first")
        with torch.cuda.device(self.device):
            cabi.check(self._lib.pbg_score_triplets_host_ids(
                self._h, _ptr(node_emb), node_emb.shape[0], _ptr(rel_w), rel_w.shape[0], _ptr(triplets_host),
                _ptr(out_block_host), B, precision_code(precision)), self._h)
