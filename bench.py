#!/usr/bin/env python
"""bench.py -- throughput of the PRO-B-GAN inference hot path (generator forward + discriminator scoring).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config base|wide] [--per-gpu-batch B]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A *step* is one canonical generator + discriminator pass (ProtBGANInference.score_triplets,
pro_b_gan_infer.py:186-209, at the tensor boundary) over one batch of synthetic triplets:
gather h/r/t rows -> G(h, r, z) -> cosine(pred, t) -> D(h, r, t) -> sigmoid.  One sample = one triplet.

Workloads (BASELINE.json):
  --config base  configs[2] at N = 1 (bf16, 4096 triplets on one B200), configs[3] at N = 8 (32768 over 8 GPUs);
                 `--per-gpu-batch 32768 / N` gives configs[3]'s literal split at N = 2 / 4.   E=128 Z=64 H=1024.
  --config wide  configs[4]: the width-scaled model (E=256, H=4096), 8192 triplets over 8 GPUs = 1024 per GPU.
Weak scaling: B triplets per GPU per step, batch-index sharded, outputs re-assembled on every rank at N > 1.

Timed region (SURVEY.md 8d "steady state: >= 100 back-to-back forward calls"; VERDICT r1 "next" #1):
  * requests are independent, so they are kept in flight on `--lanes` lanes -- one engine (ctx), one compute stream
    and one ingest stream per lane; lane l's passes occupy about a third of the SMs (50 / 50 / 48) and run beside the
    other lanes' passes; every pass also gathers (+ concatenates + casts) the lane's NEXT request into the ctx's other
    staging slot with its idle epilogue warps (pbg_score_staged_stage_next; `--stage-ahead 0`: each pass gathers its
    own request first, pbg_score_triplets);
  * inputs rotate over a pool of pre-staged batches larger than L2; every pool entry is executed once before timing;
  * each lane's rotation over its pool entries is ONE CUDA graph; the timed region replays the lanes' graphs
    back to back: exactly `steps` passes (step j runs pool entry j mod pool size) inside one CUDA-event pair, issued
    behind a short spin kernel so that the region times the GPU and not the host's launches; the region is measured
    `trials` times and the MEDIAN is the headline (`best` beside it).  A short region includes the ramp and the tail
    of the lanes: pick `steps` large enough for the figure wanted (a 4096-triplet step took ~24 us on a B200 at its
    1000 W power limit, DESIGN.md section 4);
  * `--dump-outputs DIR` writes what the last timed step returned (gen_out, gen_scores, logits, probs; float32 .npy):
    the inputs depend only on the arguments, so two builds can be compared output for output;
  * NVML clocks are sampled every 10 ms during the trials by a thread that does nothing else.

Printed JSON (one line, rank 0):
  value      samples/s, whole job, inputs resident in HBM, CUDA events, max over ranks
  e2e        same metric through the C-ABI host entry point pbg_score_triplets_host_packed (synchronous), one host thread
             per lane: per step H2D of the triplets + latents from pinned host memory and D2H of what the
             reference's score_triplets returns (pro_b_gan_infer.py:204-209)
  roofline   dominant kernel vs the measured bf16 tensor peak (MEASURED_PEAKS.json)
  cpu_baseline          the CPU oracle (a port: the reference ships no model) on the box's host cores
  gpu_library_baseline  the same oracle modules as torch bf16 on the same B200 (cuBLASLt), eager and CUDA-graphed:
             the library path this kernel has to beat (SURVEY.md:119, :433)
`--impl reference` times the CPU oracle alone as the reference arm (the reference is CPU PyTorch code).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import sys
import time
from pathlib import Path

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # lanes x (compute + ingest) streams: no false serialisation
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from

ROOT = Path(__file__).resolve().parent
for p in (str(ROOT / "pro-b-gan_b200"), str(ROOT)):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

NUM_ENTITIES, NUM_RELATIONS = 65536, 64
L2_BYTES = 126 * 2 ** 20
DUMP_MAX_BYTES = 64 * 2 ** 20
DUMP_SAMPLE_SEED = 2024
SPIN_CYCLES = 2_000_000   # ~1 ms of SM clock: longer than the host takes to issue the first launches of a region
SUSTAINED_MIN_MS = 25.0   # timed regions at least this long are compared with the sustained (power-capped) peak
METRIC = "generator+discriminator samples/sec (score_triplets pass, bf16 tensor-core mode)"
CONFIGS = {
    "base": {"E": 128, "Z": 64, "H": 1024, "batch": 4096,
             "what": "BASELINE configs[2] per GPU; configs[3] at 8 GPUs"},
    "wide": {"E": 256, "Z": 64, "H": 4096, "batch": 1024,
             "what": "BASELINE configs[4]: width-scaled model, 8192 triplets over 8 GPUs = 1024 per GPU"},
}


def flops_per_sample(E: int, Z: int, H: int) -> tuple[int, int]:
    """2*K*N per Linear (SURVEY.md 8d): base G 3 014 656, D 1 836 032; wide G 40 370 176, D 23 072 768."""
    g = 2 * ((2 * E + Z) * H + H * H + H * E)
    d = 2 * (3 * E * H + H * (H // 2) + (H // 2) * 1)
    return g, d


def measured_peaks() -> dict:
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        d = json.loads(f.read_text())
        return {"bf16_burst": d["bf16_tflops"], "bf16_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "hbm_gbs": d["hbm_gbs"], "source": "measured (MEASURED_PEAKS.json)"}
    return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm_gbs": 6650.0,
            "source": "fallback (B200_PROFILING.md)"}


def workload_name(cfg: dict, batch: int, world: int, arith: str) -> str:
    return (f"score_triplets G+D pass, {arith}, {batch} triplets/GPU/step x {world} GPU = {batch * world} per step "
            f"({cfg['what']}), E={cfg['E']} Z={cfg['Z']} H={cfg['H']}, "
            f"{NUM_ENTITIES} entities, {NUM_RELATIONS} relations")


def make_models(cfg: dict, gen_cls, disc_cls):
    from pbg import synth
    if cfg["H"] == 1024:
        return synth.make_models(gen_cls, disc_cls, cfg["E"], cfg["Z"], cfg["H"])
    return synth.make_models(gen_cls, disc_cls, cfg["E"], cfg["Z"], cfg["H"], cfg["H"])


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes {name: tensor, one row per triplet} as out_dir/<name>.npy in float32.  Above DUMP_MAX_BYTES the same
    fixed, seeded sample of rows is kept in every array, and the row numbers go to rows.npy (float64)."""
    import numpy as np
    arrays = {k: v.detach().float().cpu() for k, v in arrays.items()}
    rows = next(iter(arrays.values())).shape[0]
    row_bytes = sum(v[:1].numel() * 4 for v in arrays.values())
    if rows * row_bytes > DUMP_MAX_BYTES:
        keep = (DUMP_MAX_BYTES - 128 * (len(arrays) + 1)) // (row_bytes + 8)   # 128 B per .npy header, 8 B per row number
        idx = torch.randperm(rows, generator=torch.Generator().manual_seed(DUMP_SAMPLE_SEED))[:keep].sort().values
        arrays = {k: v[idx] for k, v in arrays.items()}
        arrays["rows"] = idx.double()
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for k, v in arrays.items():
        np.save(d / f"{k}.npy", v.numpy())


OUTPUT_NAMES = ("gen_out", "gen_scores", "logits", "probs")


# ------------------------------------------------------------------------------------------ CPU oracle leg
def cpu_oracle_pass_factory(cfg: dict, batch: int):
    """Returns (fn, cores): fn() runs one oracle G+D pass over `batch` triplets on the CPU (fp32, all threads)."""
    import torch.nn.functional as F
    from oracle import prot_b_gan_oracle as oracle  # checker / baseline only, never the product path
    from pbg import synth
    G, D = make_models(cfg, oracle.ModularGenerator, oracle.ModularDiscriminator)
    node_emb, rel_w = synth.make_tables(NUM_ENTITIES, NUM_RELATIONS, cfg["E"])
    rel_emb = torch.nn.Embedding(NUM_RELATIONS, cfg["E"])
    rel_emb.load_state_dict({"weight": rel_w})
    trip, z = synth.make_triplets(batch), synth.make_latents(batch, cfg["Z"])

    def fn():
        with torch.no_grad():
            h, r, t = node_emb[trip[:, 0]], rel_emb(trip[:, 1]), node_emb[trip[:, 2]]   # :186-188
            pred = G(h, r, z)                                                            # :201
            cs = F.cosine_similarity(pred, t, dim=1)                                     # :202
            logits, probs = D.score_triplets(node_emb, rel_emb, trip)                    # :207
        return pred, cs, logits, probs

    return fn, torch.get_num_threads()


def time_cpu_oracle(cfg: dict, batch: int, budget_s: float, max_reps: int = 200):
    fn, cores = cpu_oracle_pass_factory(cfg, batch)
    fn()  # warm-up (thread pool, allocator)
    t0 = time.perf_counter()
    reps = 0
    while reps < max_reps and (time.perf_counter() - t0 < budget_s or reps < 3):
        fn()
        reps += 1
    dt = time.perf_counter() - t0
    return batch * reps / dt, cores, reps, dt


def run_reference(args, cfg: dict, rank: int, world: int) -> None:
    """Reference arm: the reference's own implementation of the path is CPU PyTorch; its model module is not
    shipped, so the oracle port is what runs (kind = "port").  Rank 0 only."""
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)  # torchrun exports OMP_NUM_THREADS=1; the reference arm gets every core
    fn, cores = cpu_oracle_pass_factory(cfg, args.batch)
    t0 = time.perf_counter(); fn(); t_one = time.perf_counter() - t0
    # bound the whole run to ~2 minutes: shrink the per-step sample if K full batches would take longer
    sample = args.batch
    total = (args.steps + args.warmup) * t_one
    if total > 120.0:
        sample = max(256, int(args.batch * 120.0 / total) // 256 * 256)
        fn, cores = cpu_oracle_pass_factory(cfg, sample)
    for _ in range(args.warmup):
        fn()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = fn()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(OUTPUT_NAMES, res)))
    value = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(cfg, args.batch, world, "fp32 on the host CPU (the reference's arithmetic)"),
                   "device": "cpu"},
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} triplets per step x {args.steps} steps, torch {torch.__version__} fp32, "
                                   f"{cores} threads of {os.cpu_count()} logical cores"},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ torch-library leg
def time_gpu_library(cfg: dict, batch: int, dev, node_emb, rel_w) -> dict:
    """The oracle modules as torch bf16 on this GPU (cuBLASLt GEMMs + ATen elementwise / index kernels): the same
    score_triplets pass at the tensor boundary -- index gathers, G, cosine, D, sigmoid -- eager and CUDA-graphed,
    single stream and 4 graphs on 4 streams.  Checker-side code: imports oracle/, never part of the product path."""
    import torch.nn.functional as F
    from oracle import prot_b_gan_oracle as oracle
    from pbg import synth
    G, D = make_models(cfg, oracle.ModularGenerator, oracle.ModularDiscriminator)
    G, D = G.to(dev).bfloat16(), D.to(dev).bfloat16()
    nb, rb = node_emb.bfloat16(), rel_w.bfloat16()          # model state, converted once
    n_in = 8
    trips = [synth.make_triplets(batch, NUM_ENTITIES, NUM_RELATIONS, seed=700 + i).to(dev) for i in range(n_in)]
    zs = [synth.make_latents(batch, cfg["Z"], seed=800 + i).to(dev) for i in range(n_in)]

    def one(i: int):
        trip, z = trips[i % n_in], zs[i % n_in]
        h, r, t = nb[trip[:, 0]], rb[trip[:, 1]], nb[trip[:, 2]]
        pred = G(h, r, z.bfloat16())
        cs = F.cosine_similarity(pred.float(), t.float(), dim=1)
        logits = D(h, r, t).float()
        return pred, cs, logits, torch.sigmoid(logits)

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        return batch * n / (e0.elapsed_time(e1) * 1e-3)

    res = {"unit": "samples/s", "dtype": "bf16", "what": "oracle modules .to(cuda).bfloat16(), torch " + torch.__version__}
    with torch.no_grad():
        for i in range(10):
            one(i)
        n = 200
        res["eager"] = timed(lambda: [one(i) for i in range(n)], n)
        side = torch.cuda.Stream(dev)
        g = torch.cuda.CUDAGraph()
        per = 40
        with torch.cuda.stream(side):
            for i in range(3):
                one(i)
            side.synchronize()
            with torch.cuda.graph(g, stream=side):
                for i in range(per):
                    one(i)
        g.replay(); torch.cuda.synchronize()
        res["cuda_graph"] = timed(lambda: [g.replay() for _ in range(10)], per * 10)
        # 4 independent graphs on 4 streams (the same "requests in flight" policy the product uses)
        streams = [torch.cuda.Stream(dev) for _ in range(4)]
        graphs = []
        for s in streams:
            gg = torch.cuda.CUDAGraph()
            with torch.cuda.stream(s):
                one(0); s.synchronize()
                with torch.cuda.graph(gg, stream=s):
                    for i in range(per):
                        one(i)
            graphs.append(gg)
        torch.cuda.synchronize()

        def multi():
            main = torch.cuda.current_stream(dev)
            e = torch.cuda.Event(); e.record(main)
            for s, gg in zip(streams, graphs):
                s.wait_event(e)
                with torch.cuda.stream(s):
                    for _ in range(5):
                        gg.replay()
                e2 = torch.cuda.Event(); e2.record(s); main.wait_event(e2)
        multi(); torch.cuda.synchronize()
        res["cuda_graph_4_streams"] = timed(multi, per * 5 * 4)
        # The five GEMMs of one pass ALONE (cuBLASLt bf16 on these very shapes: no gather, bias, activation, cosine, hand-off),
        # 4 graphs on 4 streams, regions of >= 60 ms, first region dropped: the library's sustained rate for this pass's
        # matmuls -- the shape-limited ceiling beside MEASURED_PEAKS.json's 8192^3 figure (tools/bench_gemm_shapes.py).
        E_, Z_, H_, HD_ = cfg["E"], cfg["Z"], cfg["H"], cfg.get("HD", cfg["H"])
        shapes = [(2 * E_ + Z_, H_), (3 * E_, HD_), (H_, H_), (HD_, HD_ // 2), (H_, E_)]
        g2 = []
        for s_ in streams:
            xs = [torch.randn(batch, k, device=dev, dtype=torch.bfloat16) for k, _ in shapes]
            ws = [torch.randn(n_, k, device=dev, dtype=torch.bfloat16) for k, n_ in shapes]
            os_ = [torch.empty(batch, n_, device=dev, dtype=torch.bfloat16) for _, n_ in shapes]
            gg = torch.cuda.CUDAGraph()
            with torch.cuda.stream(s_):
                for x, w, o in zip(xs, ws, os_):
                    torch.matmul(x, w.T, out=o)
                s_.synchronize()
                with torch.cuda.graph(gg, stream=s_):
                    for _ in range(per):
                        for x, w, o in zip(xs, ws, os_):
                            torch.matmul(x, w.T, out=o)
            g2.append((gg, xs, ws, os_))
        torch.cuda.synchronize()

        def gemms(n_rep):
            def run():
                main = torch.cuda.current_stream(dev)
                e = torch.cuda.Event(); e.record(main)
                for s_, (gg, *_) in zip(streams, g2):
                    s_.wait_event(e)
                    with torch.cuda.stream(s_):
                        for _ in range(n_rep):
                            gg.replay()
                    e2 = torch.cuda.Event(); e2.record(s_); main.wait_event(e2)
            return run
        probe = timed(gemms(2), per * 2 * 4)                                   # samples/s-equivalent
        n_rep = max(2, int(0.060 * probe / (per * 4 * batch)) + 1)
        regions = [timed(gemms(n_rep), per * n_rep * 4) for _ in range(4)]
        flop_sample = sum(2.0 * k * n_ for k, n_ in shapes)
        res["gemms_only_4_streams"] = statistics.median(regions[1:])
        res["gemms_only_tflops"] = res["gemms_only_4_streams"] * flop_sample / 1e12
        res["gemms_only_what"] = ("torch.matmul bf16 on the pass's five GEMM shapes alone (" + ", ".join(f"{batch}x{k}x{n_}" for k, n_ in shapes) +
                                  "), no gather / bias / activation / cosine: samples/s-equivalent, sustained (median of 3 regions of >= 60 ms after the first)")
    res["value"] = max(res["eager"], res["cuda_graph"], res["cuda_graph_4_streams"])
    return res


# ------------------------------------------------------------------------------------------ B200 arm
def run_b200(args, cfg: dict, rank: int, local_rank: int, world: int) -> None:
    import torch.distributed as dist
    import modular_prot_b_gan as m
    from pbg import synth, shard
    from pbg.clocks import ClockSampler

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    E, Z, H = cfg["E"], cfg["Z"], cfg["H"]
    FLOP_G, FLOP_D = flops_per_sample(E, Z, H)
    FLOP_SAMPLE = FLOP_G + FLOP_D
    B = args.batch
    Bg = B * world
    K, W = args.steps, args.warmup
    S = max(1, args.lanes)
    num_sms = torch.cuda.get_device_properties(dev).multi_processor_count
    # Lane widths: a third of the device per pass, every SM used: 148 = 50 + 50 + 48 (whole CTA pairs); any three
    # consecutive lanes fill the device.  --ctas fixes one width for every lane; --lanes 1 is one full-width stream.
    if S == 1:
        widths = [args.ctas if args.ctas > 0 else 0]
    elif args.ctas > 0:
        widths = [args.ctas] * S
    else:
        per = min(S, 3)
        base_w = (num_sms // per) // 2 * 2
        extra = (num_sms - base_w * per) // 2            # pairs left over
        tri = [base_w + (2 if i < extra else 0) for i in range(per)]
        widths = [tri[i % per] for i in range(S)]
    G, D = make_models(cfg, m.ModularGenerator, m.ModularDiscriminator)
    G, D = G.to(dev), D.to(dev)
    engines = [m.make_fused_engine(G, D, ctas=widths[i]) for i in range(S)]
    cstreams = [torch.cuda.Stream(dev) for _ in range(S)]
    istreams = [torch.cuda.Stream(dev, priority=-1) for _ in range(S)]   # ingest: small kernels, scheduled first
    node_emb, rel_w = (t.to(dev) for t in synth.make_tables(NUM_ENTITIES, NUM_RELATIONS, E))
    stage_ahead = bool(args.stage_ahead)
    for e in engines:
        e.reserve(B, "bf16", 2 if stage_ahead else 0)

    # ---- input pool: distinct pre-staged batches whose footprint exceeds L2, visited round-robin
    per_batch = B * (3 * 8 + Z * 4 + E * 2 + 3 * 4)
    P = max(8, math.ceil(1.6 * L2_BYTES / per_batch))
    P = (P + 2 * S - 1) // (2 * S) * (2 * S)   # pool entry i always runs on lane i % S; an even count per lane (2 slots)
    lo, hi = shard.shard_bounds(Bg, world, rank)
    # one contiguous result block per pool entry and rank: [gen_out bf16 B x E | scores | logits | probs fp32 B each].
    # N > 1: the blocks of all ranks for one step form that step's assembled output [world, block] on EVERY rank.
    #   exchange "mc"   (default): the buffers live in symmetric memory with an NVSwitch multicast mapping and every
    #                   pass writes its rows ONCE, with multimem.st from its epilogues; the switch replicates them into
    #                   every GPU's copy (result multicast; no collective, NVLink egress = one copy of the rows)
    #   exchange "p2p": the same buffers, one unicast store per peer from the epilogues (result mirrors) -- also the
    #                   fallback when the box offers no multicast mapping
    #   exchange "nccl": one all-gather of the block per step on a per-lane communicator (eager, no graphs)
    blk_bytes = B * (2 * E + 12)
    exchange = "none"
    peer_ptrs, mc_ptr = None, 0
    if world > 1:
        exchange = args.exchange
        if exchange in ("p2p", "mc"):
            try:
                import torch.distributed._symmetric_memory as symm_mem
                sym = symm_mem.empty(P * world * blk_bytes, dtype=torch.uint8, device=dev)
                hdl = symm_mem.rendezvous(sym, dist.group.WORLD)
                peer_ptrs = [int(x) for x in hdl.buffer_ptrs]
                mc_ptr = int(getattr(hdl, "multicast_ptr", 0) or 0)
            except Exception as ex:  # symmetric memory unavailable on this box: fall back to the collective
                if rank == 0:
                    print(f"bench.py: symmetric memory unavailable ({ex}); using the NCCL all-gather", file=sys.stderr)
                exchange = "nccl"
        # every rank must take the same path: multicast > unicast mirrors > NCCL all-gather
        level = {"mc": 2 if mc_ptr else 1, "p2p": 1, "nccl": 0}[exchange]
        flag = torch.tensor([level], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        exchange = ("nccl", "p2p", "mc")[int(flag.item())]
        if exchange == "nccl":
            peer_ptrs = None
    if exchange not in ("p2p", "mc"):
        sym = torch.empty(P * max(world, 1) * blk_bytes, dtype=torch.uint8, device=dev)
    pool, mirrors, mcasts = [], [], []
    for i in range(P):
        trip = synth.make_triplets(Bg, NUM_ENTITIES, NUM_RELATIONS, seed=4321 + i)[lo:hi].contiguous().to(dev)
        z = synth.make_latents(Bg, Z, seed=1234 + i)[lo:hi].contiguous().to(dev)
        off = (i * world + rank) * blk_bytes
        blk = sym[off:off + blk_bytes]
        f32 = blk[B * 2 * E:].view(torch.float32)
        out = {"gen_out": blk[:B * 2 * E].view(torch.bfloat16).view(B, E),
               "gen_scores": f32[0:B], "logits": f32[B:2 * B], "probs": f32[2 * B:3 * B], "block": blk,
               "assembled": sym[i * world * blk_bytes:(i + 1) * world * blk_bytes]}
        pool.append((trip, z, out))
        if exchange == "p2p":
            base = [peer_ptrs[r] + off for r in range(world) if r != rank]
            mirrors.append({"gen_out": base, "gen_scores": [b + B * 2 * E for b in base],
                            "logits": [b + B * 2 * E + 4 * B for b in base], "probs": [b + B * 2 * E + 8 * B for b in base]})
        if exchange == "mc":
            b = mc_ptr + off
            mcasts.append({"gen_out": b, "gen_scores": b + B * 2 * E, "logits": b + B * 2 * E + 4 * B, "probs": b + B * 2 * E + 8 * B})
    lane_pg = None
    if exchange == "nccl":
        # one communicator per lane: collectives of different lanes run on different streams, and NCCL requires the
        # collectives of ONE communicator to execute in the same order on every rank
        lane_pg = [dist.new_group(ranks=list(range(world)), backend="nccl") for _ in range(S)]
    use_graphs = bool(args.graphs) and exchange != "nccl"   # NCCL inside per-lane graphs hung on this pool: eager there
    kw = dict(want_gen_out=True, want_gen_scores=True, want_disc=True, out_dtype=torch.bfloat16)

    # ---- one lane's work over a list of pool entries, issued on the lane's compute (+ ingest) stream
    def lane_run(l: int, entries: list[int]) -> None:
        cs, ins, eng = cstreams[l], istreams[l], engines[l]
        if not stage_ahead:
            with torch.cuda.stream(cs):
                for e in entries:
                    trip, z, out = pool[e]
                    if exchange == "p2p":
                        eng.set_result_mirrors(**mirrors[e])
                    if exchange == "mc":
                        eng.set_result_multicast(**mcasts[e])
                    eng.score_triplets(node_emb, rel_w, trip, z, precision="bf16", out=out, **kw)
                    if exchange == "nccl":  # reassemble the outputs on every rank (north_star: NVLink all-gather)
                        dist.all_gather_into_tensor(out["assembled"], out["block"], group=lane_pg[l])
            return
        if args.stage_ahead == 2:
            # in-kernel stage-ahead: pass j gathers request j + 1 into the other slot with its idle epilogue warps
            with torch.cuda.stream(cs):
                trip0, z0, _ = pool[entries[0]]
                eng.stage_triplets(0, node_emb, rel_w, trip0, z0)
                for j, e in enumerate(entries):
                    out = pool[e][2]
                    if exchange == "p2p":
                        eng.set_result_mirrors(**mirrors[e])
                    if exchange == "mc":
                        eng.set_result_multicast(**mcasts[e])
                    nxt = None
                    if j + 1 < len(entries):
                        tn, zn, _ = pool[entries[j + 1]]
                        nxt = (node_emb, rel_w, tn, zn)
                    eng.score_staged(j & 1, out=out, stage_next=nxt, **kw)
                    if exchange == "nccl":
                        dist.all_gather_into_tensor(out["assembled"], out["block"], group=lane_pg[l])
            return
        # stage-ahead: request j + 1 is gathered on the ingest stream while request j's pass runs; two slots.
        # Everything before this call on the lane is ordered by the compute stream (the ingest stream forks from it).
        fork = torch.cuda.Event(); fork.record(cs); ins.wait_event(fork)
        pass_done = [None, None]
        for j, e in enumerate(entries):
            trip, z, out = pool[e]
            slot = j & 1
            with torch.cuda.stream(ins):
                if pass_done[slot] is not None:
                    ins.wait_event(pass_done[slot])          # the pass that last read this slot
                eng.stage_triplets(slot, node_emb, rel_w, trip, z)
                staged = torch.cuda.Event(); staged.record(ins)
            with torch.cuda.stream(cs):
                cs.wait_event(staged)
                if exchange == "p2p":
                    eng.set_result_mirrors(**mirrors[e])
                if exchange == "mc":
                    eng.set_result_multicast(**mcasts[e])
                eng.score_staged(slot, out=out, **kw)
                if exchange == "nccl":
                    dist.all_gather_into_tensor(out["assembled"], out["block"], group=lane_pg[l])
                pass_done[slot] = torch.cuda.Event(); pass_done[slot].record(cs)

    lane_entries = [[e for e in range(P) if e % S == l] for l in range(S)]

    # ---- priming: every pool entry executes once, eagerly (also sizes everything and counts launches per step)
    l0 = sum(e.launch_count for e in engines)
    for l in range(S):
        lane_run(l, lane_entries[l])
    torch.cuda.synchronize()
    for e in engines:
        e.check_indices()
    launches_per_step = (sum(e.launch_count for e in engines) - l0) / P

    # ---- one CUDA graph per lane and rotation (and one per lane for a partial rotation of `n` steps)
    def capture(entries_of_lane):
        gs = []
        for l in range(S):
            if not entries_of_lane[l]:
                gs.append(None); continue
            g = torch.cuda.CUDAGraph()
            with torch.cuda.stream(cstreams[l]):
                with torch.cuda.graph(g, stream=cstreams[l]):
                    lane_run(l, entries_of_lane[l])
            gs.append(g)
        torch.cuda.synchronize()
        return gs

    main = torch.cuda.current_stream(dev)

    def issue(n_steps: int, full_graphs, tail_graphs_for) -> None:
        """n_steps passes, round-robin over the pool from entry 0: whole rotations, then a partial one."""
        rot, rem = divmod(n_steps, P)
        e = torch.cuda.Event(); e.record(main)
        for s in cstreams:
            s.wait_event(e)
        if use_graphs:
            tails = tail_graphs_for(rem) if rem else None
            for _ in range(rot):
                for l in range(S):
                    with torch.cuda.stream(cstreams[l]):
                        full_graphs[l].replay()
            for l in range(S):
                if tails is not None and tails[l] is not None:
                    with torch.cuda.stream(cstreams[l]):
                        tails[l].replay()
        else:
            for r in range(rot):
                for l in range(S):
                    lane_run(l, lane_entries[l])
            if rem:
                for l in range(S):
                    lane_run(l, [x for x in lane_entries[l] if x < rem])
        for s in cstreams:
            e2 = torch.cuda.Event(); e2.record(s); main.wait_event(e2)

    full_graphs = capture(lane_entries) if use_graphs else None
    tail_cache: dict = {}

    def tail_graphs_for(rem: int):
        if rem not in tail_cache:
            tail_cache[rem] = capture([[x for x in lane_entries[l] if x < rem] for l in range(S)])
        return tail_cache[rem]

    # ---- warm-up (graphs executed at least once, >= W steps), then `trials` timed regions of exactly K steps
    def timed(n_steps: int) -> float:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); barrier()
        torch.cuda._sleep(SPIN_CYCLES)   # the region starts once the host has issued its first launches behind it
        ev0.record(main)
        issue(n_steps, full_graphs, tail_graphs_for)
        ev1.record(main)
        torch.cuda.synchronize(); barrier()
        return ev0.elapsed_time(ev1)

    n_timed = K
    warm_steps = max(W, 2 * P)
    if use_graphs and n_timed % P:
        tail_graphs_for(n_timed % P)   # capture outside any timed region
    timed(warm_steps)
    if n_timed % P:
        timed(n_timed % P)   # the partial rotation's graphs run once before they are timed

    trials, kernel_mhz = [], []
    with ClockSampler(local_rank, period_s=0.010) as clk:
        for _ in range(max(1, args.trials)):
            trials.append(max_over_ranks(timed(n_timed)))
            # SM clock during the last pass of every lane in this trial, measured inside the kernel (clock64 / globaltimer)
            kernel_mhz.append(round(statistics.median(e.last_pass_sm_clock() for e in engines), 1))
    for e in engines:
        e.check_indices()
    if args.dump_outputs and rank == 0:
        # the last timed step ran pool entry (K - 1) mod P; at N > 1 its assembled [world, block] rows are what every
        # rank's caller receives
        blocks = pool[(n_timed - 1) % P][2]["assembled"].view(max(world, 1), blk_bytes)
        f32 = [b[B * 2 * E:].view(torch.float32).view(3, B) for b in blocks]
        dump_outputs(args.dump_outputs, {"gen_out": torch.cat([b[:B * 2 * E].view(torch.bfloat16).view(B, E) for b in blocks]),
                                         **{name: torch.cat([x[j] for x in f32]) for j, name in enumerate(OUTPUT_NAMES[1:])}})
    ms_med, ms_best = statistics.median(trials), min(trials)
    value = Bg * n_timed / (ms_med * 1e-3)
    gpu_launches = int(round(launches_per_step * n_timed))

    # ---- N > 1: the assembled buffers must equal an all-gather of the blocks, bit for bit (fails the run otherwise)
    exchange_check = None
    if world > 1:
        torch.cuda.synchronize(); barrier()
        own = sym.view(P, world, blk_bytes)[:, rank].clone()        # what this rank computed, every pool entry
        sym.zero_()
        torch.cuda.synchronize(); barrier()
        for l in range(S):
            lane_run(l, lane_entries[l])                            # every entry once more: rows land in every window
        torch.cuda.synchronize(); barrier()
        mine = sym.view(P, world, blk_bytes)[:, rank].contiguous()
        gathered = torch.empty(world, P, blk_bytes, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(gathered.view(-1), mine.view(-1))
        ref = gathered.permute(1, 0, 2).contiguous().view(-1)
        bad = int((ref != sym).sum().item())
        repeat_ok = bool(torch.equal(mine, own))
        t = torch.tensor([bad + (0 if repeat_ok else 1)], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX)
        worst = int(t.item())
        exchange_check = ("bit-identical" if worst == 0 else f"MISMATCH ({worst} bytes)") + \
            f": {P} assembled [world, block] buffers per rank vs an NCCL all-gather of the same blocks, {exchange} exchange"
        if worst != 0:
            if rank == 0:
                print("bench.py: " + exchange_check, file=sys.stderr)
            barrier(); dist.destroy_process_group()
            raise SystemExit(3)

    # ---- e2e: host buffers through the C-ABI host entry point (synchronous: H2D, pass, D2H, one sync per call);
    #      one host thread per lane keeps `S` calls in flight, each on its own ctx, like a multi-threaded server
    import threading
    hp = []
    for i in range(min(P, 16 * S)):
        # one pinned block per request, [triplets int64 B x 3 | latents fp32 B x Z]: adjacent buffers go in one H2D copy
        blk = torch.empty(B * (3 * 8 + Z * 4), dtype=torch.uint8).pin_memory()
        trip = blk[:B * 24].view(torch.int64).view(B, 3)
        z = blk[B * 24:].view(torch.float32).view(B, Z)
        trip.copy_(synth.make_triplets(Bg, NUM_ENTITIES, NUM_RELATIONS, seed=9000 + i)[lo:hi])
        z.copy_(synth.make_latents(Bg, Z, seed=9500 + i)[lo:hi])
        hp.append(blk)
    # a synchronous call spends most of its life in PCIe copies and the completion wake-up, so the server model is
    # more calls in flight than passes fit on the device: T host threads (default one per lane; --e2e-threads), one ctx each
    # (a synchronous call spins in cudaStreamSynchronize: every caller wants a core of its own -- with 8 ranks on one box the
    # default is what the host's cores allow; PBG_HOST_SYNC=block sleeps instead and measured 79-118 M against 149 M at N = 1)
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    T = args.e2e_threads if args.e2e_threads > 0 else max(2, min(S, cores // max(world, 1)))
    for e in engines:
        e.set_result_mirrors()   # host results need no re-assembly: every rank's caller receives its own shard
        e.set_result_multicast()
    e2e_engines = engines + [m.make_fused_engine(G, D, ctas=widths[i % S]) for i in range(max(0, T - S))]
    # score_triplets returns scores / logits / probabilities, not the predicted embeddings; one pinned block per thread
    # [scores | logits | probs]: one D2H copy
    h_blocks = [torch.empty(3 * B).pin_memory() for _ in range(T)]

    def e2e_worker(lane: int, first: int, last: int):
        torch.cuda.set_device(local_rank)
        for i in range(first + lane, last, T):
            e2e_engines[lane].score_triplets_host_packed(node_emb, rel_w, hp[i % len(hp)], h_blocks[lane], B, precision="bf16")

    def e2e_run(first: int, last: int) -> float:
        ts = [threading.Thread(target=e2e_worker, args=(lane, first, last)) for lane in range(T)]
        t0 = time.perf_counter()
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    e2e_run(0, 8 * T)
    torch.cuda.synchronize(); barrier()
    probe = e2e_run(0, 16 * T) / (16 * T)                      # seconds per step, all threads busy
    Ke = int(max(K, min(20000, math.ceil(args.e2e_min_s / max(probe, 1e-7)))))
    if world > 1:
        t = torch.tensor([Ke], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); Ke = int(t.item())
    Ke = (Ke + T - 1) // T * T
    torch.cuda.synchronize(); barrier()
    e2e_s = max_over_ranks(e2e_run(0, Ke))  # every call returns after the D2H of its results
    barrier()
    e2e = {"value": Bg * Ke / e2e_s, "unit": "samples/s",
           "h2d_bytes_per_step": B * (3 * 8 + Z * 4) * world, "d2h_bytes_per_step": B * 3 * 4 * world,
           "steps": Ke, "seconds": e2e_s,
           "api": f"pbg_score_triplets_host_packed (C ABI, pinned host blocks [triplets | z] in and [scores | logits | probs] out: one copy per direction, one sync per call), "
                  f"{T} host thread(s) per rank ({cores} host cores, {world} rank(s)), one ctx each; wall clock over {Ke} calls (>= --steps, long enough for "
                  f"{args.e2e_min_s} s)"}

    # ---- roofline of the dominant kernel: per-kernel CUDA events on its launch stream, the same lanes in flight
    peaks = measured_peaks()
    for e in engines:
        e.profile_enable(True); e.profile_read()
    ev = torch.cuda.Event(); ev.record(main)
    for s in cstreams:
        s.wait_event(ev)
    for l in range(S):
        lane_run(l, lane_entries[l])
    torch.cuda.synchronize()
    prof = {}
    for e in engines:
        for k, v in e.profile_read().items():
            a = prof.setdefault(k, [0.0, 0])
            a[0] += v[0]; a[1] += v[1]
        e.profile_enable(False)
        e.set_result_mirrors()
        e.set_result_multicast()
    flops = {"pass": B * FLOP_SAMPLE}  # the fused kernel runs the whole G + D pass
    kinds = {k: {"ms_per_launch": v[0] / v[1], "launches": v[1]} for k, v in prof.items() if v[1] > 0}
    dom = "pass"
    ach = flops[dom] / (kinds[dom]["ms_per_launch"] * 1e-3) / 1e12
    step_tflops = FLOP_SAMPLE * value / world / 1e12
    # Denominator (B200_PROFILING.md: "the burst figure for a kernel timed alone, the sustained one for a kernel timed
    # inside a long step"): the timed region is `steps` back-to-back passes, its length follows --steps.  When it lasts
    # at least SUSTAINED_MIN_MS and NVML reports the power cap during it (SM clocks below the maximum), the sustained
    # cuBLAS figure is the like-for-like peak; a shorter region runs mostly before the cap lowers the clock, so the
    # burst figure is.  Both fractions are always printed, and peak_source says which one `frac` uses.
    clock_summary = clk.summary()
    clock_summary["sm_mhz_in_kernel_by_trial"] = kernel_mhz   # clock64 / globaltimer over a pass's lifetime (pbg_last_pass_sm_clock)
    capped = "sw_power_cap" in (clock_summary.get("reasons") or [])
    use_sustained = capped and ms_med >= SUSTAINED_MIN_MS
    peak = peaks["bf16_sustained"] if use_sustained else peaks["bf16_burst"]
    ctas_avg = sum((w if w > 0 else num_sms) for w in widths) / len(widths)
    share = ctas_avg / num_sms
    traffic, traffic_src = None, None
    tf = ROOT / "profiles" / "traffic.json"
    if tf.exists():
        tj = json.loads(tf.read_text())
        mode = "stage2" if args.stage_ahead == 2 else "fused"
        traffic = tj.get(f"{dom}_{args.config}", tj.get(f"{dom}_{mode}", tj.get(dom)) if args.config == "base" else None)
        traffic_src = tj.get("source")
    roofline = {"bound": "tensor", "kernel": dom, "achieved": step_tflops, "peak": peak, "unit": "TFLOP/s",
                "frac": step_tflops / peak, "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peaks["source"] + (", SUSTAINED figure (cuBLAS bf16 back to back for seconds under the power cap): this "
                                                  f"timed region is {ms_med:.0f} ms x {len(trials)} trials and NVML reported sw_power_cap during it"
                                                  if use_sustained else f", burst figure (cuBLAS bf16 8192^3, best of 10): this timed "
                                                  f"region is {ms_med:.1f} ms" + ("" if capped else " and NVML reported no sw_power_cap")),
                "frac_of_burst": step_tflops / peaks["bf16_burst"], "frac_of_sustained": step_tflops / peaks["bf16_sustained"],
                "best_trial_frac_of_burst": FLOP_SAMPLE * (Bg * n_timed / (ms_best * 1e-3)) / world / 1e12 / peaks["bf16_burst"],
                "note": f"achieved = algorithmic flops per sample x measured throughput of the timed region (median "
                        f"trial) = flops of the launches in flight / their average duration x overlap; one launch "
                        f"alone: see per_launch (it occupies {ctas_avg:.0f} of {num_sms} SMs)",
                "flops_per_launch": flops[dom], "us_per_launch": kinds[dom]["ms_per_launch"] * 1e3,
                "per_launch": {"achieved": ach, "sm_share": share, "peak_share": peak * share, "frac_of_share": ach / (peak * share)},
                "whole_step": {"achieved": step_tflops, "frac": step_tflops / peaks["bf16_burst"],
                               "frac_of_sustained": step_tflops / peaks["bf16_sustained"],
                               "flops_per_sample": FLOP_SAMPLE},
                "per_kernel_us": {k: round(v["ms_per_launch"] * 1e3, 3) for k, v in kinds.items()}}

    lib = None
    if rank == 0 and world == 1 and not args.no_library_baseline:
        lib = time_gpu_library(cfg, B, dev, node_emb, rel_w)
        if lib.get("gemms_only_tflops"):
            # cuBLASLt on this pass's own GEMM shapes, same box, same power state: the shape-limited library rate
            roofline["library_gemms_only_tflops"] = lib["gemms_only_tflops"]
            roofline["frac_of_library_gemms_only"] = step_tflops / lib["gemms_only_tflops"]

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            v, cores, reps, dt = time_cpu_oracle(cfg, B, budget_s=12.0)
            cpu = {"value": v, "unit": "samples/s", "cores": cores, "kind": "port",
                   "sample": f"{reps} passes of {B} triplets in {dt:.1f} s, oracle fp32, torch {torch.__version__}, "
                             f"{cores} threads of {os.cpu_count()} logical cores"}
        line = {
            "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_med / n_timed, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "trials_ms": [round(x, 4) for x in trials], "best": Bg * n_timed / (ms_best * 1e-3),
            "config": {"workload": workload_name(cfg, B, world, "bf16"), "global_batch": Bg, "parallelism": f"dp{world}",
                       "timed_region": f"{n_timed} passes in one CUDA-event pair ({ms_med:.1f} ms"
                                       + (", short: includes the lanes' ramp and tail" if ms_med < SUSTAINED_MIN_MS else "")
                                       + f"), median of {len(trials)} trials; warm-up ran "
                                       f"{warm_steps} + {n_timed % P} steps after every pool entry had executed once",
                       "l2": f"inputs rotate over {P} distinct pre-staged batches ({P * per_batch / 2**20:.0f} MiB "
                             f"> 126 MiB L2); no flush", "cuda_graphs": bool(use_graphs),
                       "lanes": S, "ctas_per_pass": [w if w > 0 else num_sms for w in widths[:min(S, 3)]],
                       "stage_ahead": int(args.stage_ahead),
                       "collective": {"none": "none", "p2p": "none: every pass writes its result rows into all peers' symmetric-memory "
                                      "windows from its epilogues (NVLink stores, one per peer)",
                                      "mc": "none: every pass writes its result rows once, with multimem.st to the NVSwitch multicast "
                                            "address of the symmetric result buffers, from its epilogues",
                                      "nccl": "all-gather of outputs (NCCL, one per step)"}[exchange]},
            "clocks": clock_summary, "e2e": e2e, "gpu_launches": gpu_launches, "roofline": roofline,
            "cpu_baseline": cpu, "gpu_library_baseline": lib,
        }
        if exchange_check is not None:
            line["exchange_check"] = exchange_check
        print(json.dumps(line), flush=True)
    barrier()
    if world > 1:
        dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000, help="timed passes per trial (the default is a region of ~50 ms)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--config", choices=sorted(CONFIGS), default="base")
    ap.add_argument("--per-gpu-batch", "--batch", dest="batch", type=int, default=0, help="triplets per GPU per step (0: the config's)")
    ap.add_argument("--graphs", type=int, default=1)
    ap.add_argument("--lanes", type=int, default=6, help="independent requests in flight (one ctx + compute/ingest stream each)")
    ap.add_argument("--stage-ahead", type=int, default=2, help="2 (default): every pass gathers the lane's NEXT request with its idle "
                    "epilogue warps (pbg_score_staged_stage_next: +6 %% samples per SM clock, +2 %% under the power cap); 0: the pass "
                    "gathers its own request first (pbg_score_triplets); 1: the next request of a lane is staged by a separate kernel "
                    "(pbg_stage_triplets) on an ingest stream while the current pass runs")
    ap.add_argument("--exchange", choices=["mc", "p2p", "nccl"], default="mc", help="N > 1: how the outputs are re-assembled")
    ap.add_argument("--e2e-threads", type=int, default=0, help="host threads of the e2e leg (0: one per lane)")
    ap.add_argument("--e2e-min-s", type=float, default=0.4, help="the e2e leg runs at least this long (and >= --steps calls)")
    ap.add_argument("--ctas", type=int, default=0, help="SMs per pass (0: 50 / 50 / 48 of 148, whole CTA pairs)")
    ap.add_argument("--trials", type=int, default=5, help="timed regions of --steps steps each; the median is the headline")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step returned to DIR/<name>.npy (float32, at most 64 MiB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        raise SystemExit("bench.py: --steps must be >= 1")
    cfg = CONFIGS[args.config]
    if args.batch <= 0:
        args.batch = cfg["batch"]
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world == 1 and args.gpus > 1:
        raise SystemExit("bench.py: --gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args, cfg, rank, world)
    else:
        run_b200(args, cfg, rank, local_rank, world)


if __name__ == "__main__":
    main()
