"""Fused host for the inference entry points: the methods of the reference's ``ProtBGANInference`` class
(pro_b_gan_infer.py:43-338) re-stated over the C ABI, one launch per request instead of one torch op per line.

Two ways to run on these kernels:
  * keep the reference script and inject ``modular_prot_b_gan`` (``pbg.launcher``): module-by-module drop-in, the
    script's own gathers / cosine / top-k stay torch ops;
  * use this class (same constructor arguments, method names, argument meaning, result dictionaries and error types):
        score_triplets        :167-211  ->  ONE fused pass (gather + G + cosine + D), host buffers in / out
        predict_tails         :118-165  ->  gather + G in one launch, then the entity scorer (no [B, N] matrix)
        find_similar_entities :213-263  ->  the entity scorer on gathered rows
        analyze_relations     :265-318  ->  one discriminator pass over all head x tail x relation triplets
        get_model_info        :322-338
    Inputs may be the reference's Python lists, the CLI's JSON text (parsed in C, pbg.hostio), ndarrays or tensors.

Checkpoint format = the reference's (:74-116): ``args`` {embed_dim, noise_dim, hidden_dim}, ``node_emb`` [N, E],
``rel_emb`` {weight [R, E]}, ``generator`` / ``discriminator`` state dicts, optional ``best_val_hit10``, ``best_epoch``,
``training_history``.  BatchNorm folding + bf16 packing happen once here, at load.  CUDA only: no CPU path."""
from __future__ import annotations

import os
import time
from typing import Any, Dict

import numpy as np
import torch

from . import hostio
from .analyze import analyze_relations_batched


class FusedInference:
    def __init__(self, checkpoint_path: str, device: str = "auto", precision: str | None = None, verbose: bool = False,
                 latents: str | None = None):
        """``latents``: 'cpu' (default; PBG_LATENTS overrides) draws z from the generator's CPU mt19937 stream, as the
        oracle does, and ships it with the ids; 'cuda' draws z on the device from a Philox stream seeded LATENT_SEED
        (what torch.randn(..., device='cuda', generator=g) gives), so only ids cross PCIe."""
        import modular_prot_b_gan as m
        if device in ("auto", "cuda"):
            if not torch.cuda.is_available():
                raise RuntimeError("pro-b-gan_b200 has no CPU path: a CUDA (sm_100a) device is required")
            self.device = torch.device("cuda", torch.cuda.current_device())
        else:
            self.device = torch.device(device)
            if self.device.type != "cuda":
                raise RuntimeError(f"device {device!r}: pro-b-gan_b200 has no CPU path")
        self.checkpoint_path = checkpoint_path
        self.precision = precision
        if not os.path.exists(checkpoint_path):
            raise FileNotFoundError(f"Checkpoint not found: {checkpoint_path}")     # :71-72
        t0 = time.perf_counter()
        ckpt = torch.load(checkpoint_path, map_location="cpu")
        t1 = time.perf_counter()
        args = ckpt.get("args", {})
        if not isinstance(args, dict):
            args = vars(args)
        self.embed_dim = args.get("embed_dim", 128)                                 # defaults of :77-80
        self.noise_dim = args.get("noise_dim", 64)
        self.hidden_dim = args.get("hidden_dim", 1024)
        self.node_emb = ckpt["node_emb"].detach().to(self.device, torch.float32).contiguous()
        self.rel_weight = ckpt["rel_emb"]["weight"].detach().to(self.device, torch.float32).contiguous()
        self.num_entities, self.num_relations = int(self.node_emb.shape[0]), int(self.rel_weight.shape[0])
        self.generator = m.ModularGenerator(self.embed_dim, self.noise_dim)
        self.discriminator = m.ModularDiscriminator(self.embed_dim, self.hidden_dim)
        self.generator.load_state_dict(ckpt["generator"])                           # strict, like :97-98
        self.discriminator.load_state_dict(ckpt["discriminator"])
        self.generator.to(self.device).eval()
        self.discriminator.to(self.device).eval()
        self.generator.precision = self.discriminator.precision = precision
        t2 = time.perf_counter()
        self.engine = m.make_fused_engine(self.generator, self.discriminator)       # BN fold + bf16 pack + upload
        self.latents = m.latent_source(latents)
        if self.latents == "cuda":
            self.engine.set_latent_stream(True, m.LATENT_SEED, 0)
        torch.cuda.synchronize(self.device)
        t3 = time.perf_counter()
        self.best_val_hit10 = ckpt.get("best_val_hit10", 0.0)
        self.best_epoch = ckpt.get("best_epoch", 0)                                   # :111
        self.training_history = ckpt.get("training_history", {})
        self.ingest_ms = {"torch_load": (t1 - t0) * 1e3, "tables_and_modules": (t2 - t1) * 1e3,
                          "fold_pack_upload": (t3 - t2) * 1e3}
        self._pinned: Dict[str, torch.Tensor] = {}
        if verbose:
            print(f"FusedInference ready: {self.num_entities:,} entities, {self.num_relations:,} relations, "
                  f"E={self.embed_dim}; ingest {self.ingest_ms}")

    def reseed(self, seed: int | None = None) -> None:
        """Restart the latent stream this object draws from (CPU generator or device stream) at `seed`."""
        import modular_prot_b_gan as m
        seed = m.LATENT_SEED if seed is None else int(seed)
        self.generator.reseed(seed)
        if self.latents == "cuda":
            self.engine.set_latent_stream(True, seed, 0)

    # ------------------------------------------------------------------ helpers
    def _pin(self, name: str, rows: int, shape_tail: tuple, dtype) -> torch.Tensor:
        """Grow-only pinned staging buffer; returns the first `rows` rows."""
        buf = self._pinned.get(name)
        if buf is None or buf.shape[0] < rows or buf.dtype != dtype or tuple(buf.shape[1:]) != tuple(shape_tail):
            cap = max(256, 1 << max(rows - 1, 1).bit_length())
            buf = self._pinned[name] = torch.empty((cap, *shape_tail), dtype=dtype, pin_memory=True)
        return buf[:rows]

    def _stage_rows(self, name: str, x, cols: int) -> torch.Tensor:
        rows = hostio.index_rows(x, cols)
        buf = self._pin(name, rows.shape[0], (cols,), torch.int64)
        buf.copy_(rows)
        return buf

    def _latents(self, batch: int) -> torch.Tensor:
        """The generator's own latent draw (CPU mt19937 stream of the module, bit-exact with the oracle), written
        straight into pinned memory."""
        buf = self._pin("z", batch, (self.noise_dim,), torch.float32)
        if batch:
            torch.randn(batch, self.noise_dim, generator=self.generator._latent_gen, dtype=torch.float32, out=buf)
        return buf

    @staticmethod
    def _echo(x, rows: torch.Tensor, flat: bool = False):
        """The reference echoes the caller's own list in its result; text / array inputs are echoed as lists."""
        if isinstance(x, (list, tuple)):
            return x
        return rows[:, 0].tolist() if flat else rows.tolist()

    # ------------------------------------------------------------------ :167-211
    def score_triplets(self, triplets, method: str = "both", as_arrays: bool = False) -> Dict[str, Any]:
        """``as_arrays=True`` returns numpy arrays instead of Python lists (same keys, same values): no ``.tolist()``,
        and ``pbg.hostio.dumps_results`` writes them as the JSON text json.dumps would print for the lists."""
        trip = self._stage_rows("trip", triplets, 3)
        B = trip.shape[0]
        out = (lambda t: t.numpy().copy()) if as_arrays else (lambda t: t.tolist())   # staging buffers are reused
        results: Dict[str, Any] = {
            "triplets": trip.numpy().copy() if as_arrays else self._echo(triplets, trip),
            "metadata": {"num_triplets": B, "method": method, "model_hit10": self.best_val_hit10},
        }
        if B == 0:
            raise IndexError("too many indices for tensor of dimension 1")   # torch.tensor([])[:, 0] at :183
        run_g, run_d = method in ("generator", "both"), method in ("discriminator", "both")
        if not (run_g or run_d):
            return results                                   # an unknown method yields metadata only, as :196-209
        if self.latents == "cuda" and run_g and run_d:
            # only the ids travel: [triplets] in, [gen_scores | logits | probs] out, latents drawn on the device
            block = self._pin("out_block", 3 * B, (), torch.float32)
            scores, logits, probs = block[:B], block[B:2 * B], block[2 * B:]
            with torch.cuda.device(self.device):
                self.engine.score_triplets_host_ids(self.node_emb, self.rel_weight, trip, block, precision=self.precision)
        else:
            z = self._latents(B) if run_g and self.latents == "cpu" else None
            scores = self._pin("gen_scores", B, (), torch.float32) if run_g else None
            logits = self._pin("logits", B, (), torch.float32) if run_d else None
            probs = self._pin("probs", B, (), torch.float32) if run_d else None
            with torch.cuda.device(self.device):
                self.engine.score_triplets_host(self.node_emb, self.rel_weight, trip, z, None, scores, logits, probs,
                                                precision=self.precision)   # raises IndexError on a bad id
        if run_g:
            results["generator_scores"] = out(scores)
        if run_d:
            results["discriminator_logits"] = out(logits)
            results["discriminator_probabilities"] = out(probs)
        return results

    # ------------------------------------------------------------------ :118-165
    def predict_tails(self, head_relation_pairs, top_k: int = 10, return_scores: bool = False,
                      as_arrays: bool = False) -> Dict[str, Any]:
        pairs = self._stage_rows("pairs", head_relation_pairs, 2)
        out = (lambda t: t.cpu().numpy()) if as_arrays else (lambda t: t.tolist())
        B = pairs.shape[0]
        self.engine.validate_top_k(top_k, self.num_entities)   # before anything is launched from the reused staging buffers
        with torch.no_grad(), torch.cuda.device(self.device):
            try:
                dev_pairs = pairs.to(self.device, non_blocking=True)
                z = self._latents(B).to(self.device, non_blocking=True) if self.latents == "cpu" else None
                pred = self.engine.generator_forward_gather(self.node_emb, self.rel_weight, dev_pairs[:, 0], dev_pairs[:, 1],
                                                            z, precision=self.precision)
                top_scores, top_idx = self.engine.cosine_topk(pred, self.node_emb, top_k)
                self.engine.check_indices()
            except BaseException:
                torch.cuda.current_stream(self.device).synchronize()   # the copies out of the pinned buffers must not outlive the call
                raise
            results: Dict[str, Any] = {
                "predictions": out(top_idx),
                "metadata": {"num_queries": B, "top_k": top_k, "model_hit10": self.best_val_hit10},
            }
            if return_scores:
                results["scores"] = out(top_scores)
        return results

    # ------------------------------------------------------------------ :213-263
    def find_similar_entities(self, entity_ids, top_k: int = 10) -> Dict[str, Any]:
        ids = hostio.index_rows(entity_ids, 1)[:, 0]
        if ids.numel() and (int(ids.min()) < -self.num_entities or int(ids.max()) >= self.num_entities):
            raise IndexError(f"index out of range for node_emb with {self.num_entities} rows")
        echo = entity_ids if isinstance(entity_ids, (list, tuple)) else ids.tolist()
        results: Dict[str, Any] = {
            "similar_entities": [],
            "metadata": {"num_queries": int(ids.numel()), "top_k": top_k, "model_hit10": self.best_val_hit10},
        }
        self.engine.validate_top_k(top_k + 1, self.num_entities)
        with torch.no_grad(), torch.cuda.device(self.device):
            q = self.node_emb[ids.to(self.device)]
            top_scores, top_idx = self.engine.cosine_topk(q, self.node_emb, top_k + 1)
            top_scores, top_idx = top_scores.cpu().numpy(), top_idx.cpu().numpy()
        for i, query_id in enumerate(echo):
            keep = top_idx[i] != query_id                    # drop the query itself, then cut to top_k (:251-255)
            results["similar_entities"].append({
                "query_entity": query_id,
                "similar_entities": top_idx[i][keep][:top_k].tolist(),
                "similarity_scores": top_scores[i][keep][:top_k].tolist(),
            })
        return results

    # ------------------------------------------------------------------ :265-318
    def analyze_relations(self, head_entities, tail_entities, top_k: int = 5) -> Dict[str, Any]:
        heads = hostio.index_rows(head_entities, 1)[:, 0]
        tails = hostio.index_rows(tail_entities, 1)[:, 0]
        res = analyze_relations_batched(self.discriminator, self.node_emb, self.rel_weight, heads.tolist(),
                                        tails.tolist(), top_k, self.best_val_hit10)
        if isinstance(head_entities, (list, tuple)) and isinstance(tail_entities, (list, tuple)):
            it = iter(res["relation_analysis"])              # echo the caller's own objects, as the reference does
            for h in head_entities:
                for t in tail_entities:
                    e = next(it)
                    e["head_entity"], e["tail_entity"] = h, t
        return res

    # ------------------------------------------------------------------ :322-338
    def get_model_info(self) -> Dict[str, Any]:
        return {
            "model_architecture": {"embedding_dim": self.embed_dim, "noise_dim": self.noise_dim,
                                   "hidden_dim": self.hidden_dim, "num_entities": self.num_entities,
                                   "num_relations": self.num_relations},
            "training_performance": {"best_validation_hit10": self.best_val_hit10, "best_epoch": self.best_epoch},
            "checkpoint_path": self.checkpoint_path,
            "device": str(self.device),
        }
