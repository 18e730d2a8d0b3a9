"""Drop-in ``modular_prot_b_gan``: the module pro_b_gan_infer.py imports (:41) but does not ship,
with its forward passes running on hand-written sm_100a kernels through the C ABI (include/pbg.h).

Same constructor and call signatures as the reference's call sites:
  Generator(embed_dim, noise_dim)            pro_b_gan_infer.py:93      forward(h_emb, r_emb)            :143, :201
  Discriminator(embed_dim, hidden_dim)       pro_b_gan_infer.py:94      forward(h_emb, r_emb, t_emb)     :301
                                                                        score_triplets(node_emb, rel_emb, triplets) :207
Both are nn.Modules whose parameters live in stock nn.Linear / nn.BatchNorm1d containers under ``net`` so that
``.to(device)``, strict ``load_state_dict`` and ``.eval()`` (:93-98, :106-107) behave exactly like the
oracle's; the containers are never *called* -- at first forward the weights are BatchNorm-folded, packed to bf16
and handed to libpbg_b200.so, and every later forward is a C-ABI call.

No CPU fallback and no second backend: a module left on the CPU, or a box without an sm_100 GPU, raises.
Precision: ``PBG_PRECISION=bf16`` (default, tcgen05 tensor cores) or ``fp32`` (SIMT parity mode), or set the
``precision`` attribute on the module.
Latents: ``PBG_LATENTS=cpu`` (default: the oracle's CPU mt19937 stream, copied to the device) or ``cuda`` (drawn on the
device, bit for bit what ``torch.randn(..., device='cuda', generator=g)`` gives for g seeded LATENT_SEED), or set the
generator's ``latent_source`` attribute.
"""
from __future__ import annotations

import os

import torch
import torch.nn as nn

from pbg.engine import Engine, fold_linear_bn

LEAKY_SLOPE = 0.2
DEFAULT_G_HIDDEN = 1024
LATENT_SEED = 1234


class _CudaModule(nn.Module):
    precision: str | None = None   # None -> PBG_PRECISION env var -> 'bf16'
    check_indices: bool = True     # raise IndexError like the reference (costs one 4-byte D2H + sync)

    def __init__(self):
        super().__init__()
        self._engine: Engine | None = None
        self._engine_key = None

    def _state_key(self):
        ts = list(self.parameters()) + list(self.buffers())
        return tuple((t.device, t.data_ptr(), t._version) for t in ts)

    def _device(self) -> torch.device:
        return next(self.parameters()).device

    def _require_inference(self):
        if self.training:
            raise RuntimeError("pro-b-gan_b200 modules are inference-only: call .eval() first "
                               "(the reference does, pro_b_gan_infer.py:106-107)")
        dev = self._device()
        if dev.type != "cuda":
            raise RuntimeError(f"{type(self).__name__} is on {dev}: pro-b-gan_b200 has no CPU path; "
                               "move the module to an sm_100a CUDA device")

    def _get_engine(self) -> Engine:
        self._require_inference()
        key = self._state_key()
        if self._engine is None or key != self._engine_key:
            self._engine = self._build_engine()
            self._engine_key = key
        return self._engine

    def _build_engine(self) -> Engine:  # pragma: no cover - abstract
        raise NotImplementedError


def latent_source(value: str | None = None) -> str:
    """'cpu' or 'cuda': `value`, else the PBG_LATENTS env var, else 'cpu'."""
    src = (value or os.environ.get("PBG_LATENTS", "cpu")).lower()
    if src not in ("cpu", "cuda"):
        raise ValueError(f"unknown latent source {src!r}; use 'cpu' or 'cuda'")
    return src


class ModularGenerator(_CudaModule):
    latent_source: str | None = None   # None -> PBG_LATENTS env var -> 'cpu'

    def __init__(self, embed_dim: int, noise_dim: int, hidden_dim: int = DEFAULT_G_HIDDEN):
        super().__init__()
        self.embed_dim, self.noise_dim, self.hidden_dim = embed_dim, noise_dim, hidden_dim
        self.net = nn.Sequential(  # parameter containers only; same keys as the oracle's state_dict
            nn.Linear(2 * embed_dim + noise_dim, hidden_dim),
            nn.BatchNorm1d(hidden_dim),
            nn.LeakyReLU(LEAKY_SLOPE),
            nn.Linear(hidden_dim, hidden_dim),
            nn.BatchNorm1d(hidden_dim),
            nn.LeakyReLU(LEAKY_SLOPE),
            nn.Linear(hidden_dim, embed_dim),
            nn.Tanh(),
        )
        self._latent_gen = torch.Generator(device="cpu")
        self._latent_gen.manual_seed(LATENT_SEED)
        self._latent_seed = LATENT_SEED
        self._stream_engine: Engine | None = None   # the engine whose ctx holds the device latent stream

    def reseed(self, seed: int = LATENT_SEED) -> None:
        """Restart the latent stream: the CPU generator, and the device stream (at Philox offset 0) with its next draw."""
        self._latent_gen.manual_seed(seed)
        self._latent_seed = seed
        self._stream_engine = None

    def _device_stream(self) -> Engine:
        """The engine, with its ctx's latent stream on; a rebuilt engine continues where the previous one stopped."""
        eng = self._get_engine()
        if self._stream_engine is not eng:
            pos = self._stream_engine.latent_stream() if self._stream_engine is not None else (self._latent_seed, 0)
            eng.set_latent_stream(True, *pos)
            self._stream_engine = eng
        return eng

    def sample_latent(self, batch: int) -> torch.Tensor:
        if latent_source(self.latent_source) == "cuda":
            eng = self._device_stream()
            if batch == 0:
                return torch.empty(0, self.noise_dim, dtype=torch.float32, device=eng.device)
            seed, off = eng.latent_stream()
            z, after = eng.draw_latents(batch, seed, off)
            eng.set_latent_stream(True, seed, after)
            return z
        # the sampling step is bit-exact with the oracle: same CPU mt19937 stream, then one H2D copy
        return torch.randn(batch, self.noise_dim, generator=self._latent_gen, dtype=torch.float32)

    def folded_layers(self):
        n = self.net
        return [fold_linear_bn(n[0], n[1]), fold_linear_bn(n[3], n[4]), fold_linear_bn(n[6], None)]

    def _build_engine(self) -> Engine:
        eng = Engine(self.embed_dim, self.noise_dim, self.hidden_dim, 16, self._device(), LEAKY_SLOPE)
        eng.load_generator(self.folded_layers())
        return eng

    def forward(self, h_emb: torch.Tensor, r_emb: torch.Tensor, z: torch.Tensor | None = None) -> torch.Tensor:
        if z is None and latent_source(self.latent_source) == "cuda":
            return self._device_stream().generator_forward(h_emb, r_emb, None, precision=self.precision)
        eng = self._get_engine()
        if z is None:
            z = self.sample_latent(h_emb.shape[0])
        z = z.to(h_emb.device, non_blocking=True)
        return eng.generator_forward(h_emb, r_emb, z, precision=self.precision)


class ModularDiscriminator(_CudaModule):
    def __init__(self, embed_dim: int, hidden_dim: int):
        super().__init__()
        self.embed_dim, self.hidden_dim = embed_dim, hidden_dim
        self.net = nn.Sequential(
            nn.Linear(3 * embed_dim, hidden_dim),
            nn.LeakyReLU(LEAKY_SLOPE),
            nn.Linear(hidden_dim, hidden_dim // 2),
            nn.LeakyReLU(LEAKY_SLOPE),
            nn.Linear(hidden_dim // 2, 1),
        )

    def folded_layers(self):
        n = self.net
        return [fold_linear_bn(n[0], None), fold_linear_bn(n[2], None), fold_linear_bn(n[4], None)]

    def _build_engine(self) -> Engine:
        eng = Engine(self.embed_dim, 8, 8, self.hidden_dim, self._device(), LEAKY_SLOPE)
        eng.load_discriminator(self.folded_layers())
        return eng

    def forward(self, h_emb: torch.Tensor, r_emb: torch.Tensor, t_emb: torch.Tensor) -> torch.Tensor:
        logits, _ = self._get_engine().discriminator_forward(h_emb, r_emb, t_emb, precision=self.precision)
        return logits  # 1-D [B]: .item() works at B = 1 (pro_b_gan_infer.py:301)

    def score_triplets(self, node_emb: torch.Tensor, rel_emb, triplets: torch.Tensor):
        eng = self._get_engine()
        rel_w = rel_emb.weight if isinstance(rel_emb, nn.Module) else rel_emb
        res = eng.score_triplets(node_emb, rel_w, triplets, want_disc=True, precision=self.precision)
        if self.check_indices:
            eng.check_indices()
        return res["logits"], res["probs"]


def make_fused_engine(generator: ModularGenerator, discriminator: ModularDiscriminator, ctas: int = 0) -> Engine:
    """One ctx holding both models: the G + D pass of ProtBGANInference.score_triplets
    (pro_b_gan_infer.py:186-209) as a single call sharing one gather.  `ctas`: SMs per pass (0 = all); servers
    with several independent passes in flight use one engine + stream per lane at about a third of the device."""
    generator._require_inference()
    discriminator._require_inference()
    eng = Engine(generator.embed_dim, generator.noise_dim, generator.hidden_dim, discriminator.hidden_dim,
                 generator._device(), LEAKY_SLOPE, ctas)
    eng.load_generator(generator.folded_layers())
    eng.load_discriminator(discriminator.folded_layers())
    return eng


_TOPK_ENGINES: dict = {}


def cosine_topk(queries: torch.Tensor, table: torch.Tensor, k: int):
    """Drop-in for the entity-scoring lines of the reference script (pro_b_gan_infer.py:146-151 and :231-236):

        pred_norm = F.normalize(pred_emb, dim=-1); entity_norm = F.normalize(self.node_emb, dim=-1)
        similarities = torch.matmul(pred_norm, entity_norm.T); top_scores, top_indices = similarities.topk(top_k, dim=1)
    becomes
        top_scores, top_indices = modular_prot_b_gan.cosine_topk(pred_emb, self.node_emb, top_k)

    CUDA tensors only (no CPU fallback).  One scoring ctx per (device, embedding width) is kept alive."""
    if queries.device.type != "cuda" or table.device != queries.device:
        raise RuntimeError("cosine_topk runs only on CUDA tensors on one device; there is no CPU fallback")
    E = int(table.shape[1])
    key = (queries.device.index, E)
    eng = _TOPK_ENGINES.get(key)
    if eng is None:
        eng = _TOPK_ENGINES[key] = Engine(E, 8, 8, 16, queries.device, LEAKY_SLOPE)   # model dims unused by the scorer
    return eng.cosine_topk(queries.detach(), table.detach(), k)


# names the reference script instantiates (pro_b_gan_infer.py:93-94)
Generator = ModularGenerator
Discriminator = ModularDiscriminator
