"""Device latents (csrc/latent.cuh) against host latents on one GPU:
  1. the draw kernel (pbg_draw_latents) against torch.randn on the same CUDA generator, B x Z = 64;
  2. FusedInference.score_triplets / predict_tails with latents='cpu' (CPU mt19937 draw, shipped over PCIe) against
     latents='cuda' (drawn on the device), from an int64 tensor and from JSON text;
  3. end-to-end samples/s through pbg_score_triplets_host_ids (24 B in, 12 B out per sample) against
     pbg_score_triplets_host_packed (24 + 256 B in, 12 B out) from T host threads, one ctx + stream each.
python tools/bench_latents.py [--out FILE]"""
import argparse
import json
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT / "pro-b-gan_b200"), str(ROOT)]
import torch

import modular_prot_b_gan as m
from pbg import synth
from pbg.inference import FusedInference

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=None)
args = ap.parse_args()
out = open(args.out, "w") if args.out else None


def P(s):
    print(s, flush=True)
    if out:
        out.write(s + "\n"); out.flush()


def events_ms(f, n):
    """Mean device time per call over n back-to-back calls (CUDA events), after a warm-up call."""
    f(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        f()
    b.record(); b.synchronize()
    return a.elapsed_time(b) / n


def graph_us(f, n):
    """Device time per call of n calls captured into one CUDA graph (no host launch cost), median of 5 replays."""
    f(); torch.cuda.synchronize()
    g, s = torch.cuda.CUDAGraph(), torch.cuda.Stream()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            for _ in range(n):
                f()
    ts = []
    for _ in range(6):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(s):
            a.record(); g.replay(); b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b) * 1e3 / n)
    return sorted(ts[1:])[2]


def host_ms(f, n):
    """Median host time of n synchronous calls, after two warm-up calls."""
    f(); f(); torch.cuda.synchronize()
    ts = []
    for _ in range(n):
        t0 = time.perf_counter(); f(); torch.cuda.synchronize(); ts.append((time.perf_counter() - t0) * 1e3)
    return sorted(ts)[len(ts) // 2]


dev = torch.device("cuda:0")
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
P(f"device: {torch.cuda.get_device_name(dev)} | nvidia-smi: {smi} | torch {torch.__version__}")
SIZES = (4096, 32768)

# ---------------------------------------------------------------- 1. the draw
P("\n1. latent draw, [B, 64] fp32: device time per draw, 200 draws captured in one CUDA graph (median of 5 replays); "
  "and per call from Python (CUDA events over 500 eager calls, host launch cost included)")
from pbg.engine import Engine
eng = Engine(128, 64, 8, 16, dev)
g = torch.Generator(device=dev); g.manual_seed(1234)
for B in SIZES:
    z = torch.empty(B, 64, device=dev)
    t_dev = events_ms(lambda: eng.draw_latents(B, 1234, 0), 500)
    t_torch = events_ms(lambda: torch.randn((B, 64), device=dev, generator=g, out=z), 500)
    k_dev = graph_us(lambda: eng.draw_latents(B, 1234, 0), 200)
    k_torch = graph_us(lambda: torch.randn((B, 64), device=dev, out=z), 200)   # the default generator: capturable
    g.set_offset(8)
    ok = torch.equal(eng.draw_latents(B, 1234, 8)[0], torch.randn((B, 64), device=dev, generator=g))
    P(f"   B = {B:6d}: device time: pbg_draw_latents {k_dev:6.2f} us | torch.randn {k_torch:6.2f} us;  eager call: "
      f"Engine.draw_latents {t_dev * 1e3:6.2f} us (allocates its output) | torch.randn(out=) {t_torch * 1e3:6.2f} us | "
      f"bit-identical: {ok}")

# ---------------------------------------------------------------- 2. FusedInference
P("\n2. FusedInference requests (host wall time, median of 20 synchronous calls, bf16 mode)")
with tempfile.TemporaryDirectory() as d:
    path = str(Path(d) / "ckpt.pt")
    torch.save(synth.make_checkpoint(m.ModularGenerator, m.ModularDiscriminator), path)
    infs = {src: FusedInference(path, "cuda", latents=src) for src in ("cpu", "cuda")}
for B in SIZES:
    trip = synth.make_triplets(B)
    text = json.dumps(trip.tolist())
    pairs = trip[:, :2].contiguous()
    for what, f in (("score_triplets from an int64 tensor", lambda i: i.score_triplets(trip, as_arrays=True)),
                    ("score_triplets from JSON text", lambda i: i.score_triplets(text, as_arrays=True)),
                    ("predict_tails (top 10) from an int64 tensor", lambda i: i.predict_tails(pairs, 10, as_arrays=True))):
        t = {src: host_ms(lambda: f(i), 20) for src, i in infs.items()}
        P(f"   B = {B:6d} {what:45s}: cpu latents {t['cpu']:8.3f} ms | cuda latents {t['cuda']:8.3f} ms "
          f"({t['cpu'] / t['cuda']:.1f}x)")
del infs

# ---------------------------------------------------------------- 3. end to end from host threads
P("\n3. end to end, host ids in -> host results out, B = 4096 per call, bf16 mode, one ctx + stream per thread "
  "(launch width 48 SMs), 3 s per point")
G, D = synth.make_models(m.ModularGenerator, m.ModularDiscriminator)
G, D = G.to(dev).eval(), D.to(dev).eval()
node_emb, rel_w = (t.to(dev) for t in synth.make_tables())
B, Z = 4096, 64


def lane(form, stop, ready, counts, i):
    torch.cuda.set_device(dev)
    e = m.make_fused_engine(G, D, ctas=48)
    e.reserve(B, "bf16")
    trip = synth.make_triplets(B, seed=100 + i)
    outb = torch.empty(3 * B, dtype=torch.float32).pin_memory()
    if form == "ids":
        e.set_latent_stream(True, 1234 + i, 0)
        inb = trip.pin_memory()
        call = lambda: e.score_triplets_host_ids(node_emb, rel_w, inb, outb)
    else:
        inb = torch.empty(B * (24 + 4 * Z), dtype=torch.uint8).pin_memory()
        inb[:24 * B].view(torch.int64).copy_(trip.reshape(-1))
        inb[24 * B:].view(torch.float32).copy_(synth.make_latents(B, seed=i).reshape(-1))
        call = lambda: e.score_triplets_host_packed(node_emb, rel_w, inb, outb, B)
    call(); call()
    ready.wait()
    while not stop.is_set():
        call()
        counts[i] += 1


for T in (1, 3, 6):
    res = {}
    for form in ("packed", "ids"):
        stop, ready, counts = threading.Event(), threading.Barrier(T + 1), [0] * T
        th = [threading.Thread(target=lane, args=(form, stop, ready, counts, i)) for i in range(T)]
        for t in th:
            t.start()
        ready.wait(timeout=120)
        t0 = time.perf_counter()
        time.sleep(3.0)
        n = sum(counts); dt = time.perf_counter() - t0
        stop.set()
        for t in th:
            t.join()
        res[form] = n * B / dt / 1e6
    P(f"   T = {T}: _host_packed (caller latents) {res['packed']:7.2f} M samples/s | _host_ids (device latents) "
      f"{res['ids']:7.2f} M samples/s ({res['ids'] / res['packed']:.2f}x)")
