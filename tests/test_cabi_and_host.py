"""CPU tests of the boundary and the host logic: the C-ABI library loads and exports every symbol include/pbg.h
declares, fails loudly without a GPU (no CPU fallback), BatchNorm folding, module plumbing, sharding (gloo, ws=2)."""
import os
import re
import subprocess
import sys
from pathlib import Path

import pytest
import torch
import torch.nn as nn

ROOT = Path(__file__).resolve().parent.parent
HEADER = ROOT / "include" / "pbg.h"


@pytest.fixture(scope="module")
def lib():
    from pbg import build, cabi
    build.build()
    return cabi.load()


def declared_symbols() -> set[str]:
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    return set(re.findall(r"\b(pbg_[a-z0-9_]+)\s*\(", text))


def test_library_exports_every_declared_symbol(lib):
    from pbg import build, cabi
    out = subprocess.run(["nm", "-D", "--defined-only", str(build.LIB_PATH)], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (pbg_[a-z0-9_]+)", out))
    declared = declared_symbols()
    assert declared, "header parse found nothing"
    assert declared <= exported, f"declared but not exported: {sorted(declared - exported)}"
    assert exported <= declared, f"exported but not declared in include/pbg.h: {sorted(exported - declared)}"
    assert set(cabi.SYMBOLS) == declared
    for s in declared:
        assert hasattr(lib, s)


def test_abi_version(lib):
    assert lib.pbg_abi_version() == 1


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_create_fails_loudly_without_gpu(lib):
    import ctypes as C
    from pbg import cabi
    h = C.c_void_p(0)
    dims = cabi.PbgDims(128, 64, 1024, 1024, 0, 0.2)
    st = lib.pbg_create(C.byref(h), C.byref(dims))
    assert st == cabi.PBG_ERR_UNSUPPORTED and not h.value
    assert b"no CPU fallback" in lib.pbg_last_error(None)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_modules_refuse_to_run_on_cpu(synth):
    import modular_prot_b_gan as m
    G, D = synth.make_models(m.ModularGenerator, m.ModularDiscriminator)
    with pytest.raises(RuntimeError, match="no CPU path"):
        G(torch.zeros(2, 128), torch.zeros(2, 128))
    with pytest.raises(RuntimeError, match="no CPU path"):
        D(torch.zeros(2, 128), torch.zeros(2, 128), torch.zeros(2, 128))
    from pbg.engine import Engine
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        Engine(128, 64, 1024, 1024, "cpu")


def test_product_path_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under the package (or the tools) may import it."""
    for f in list((ROOT / "pro-b-gan_b200").rglob("*.py")) + list((ROOT / "tools").glob("*.py")):
        assert not re.search(r"^\s*(from|import)\s+oracle\b", f.read_text(), flags=re.M), f


def test_state_dicts_are_interchangeable(oracle, synth):
    """strict load_state_dict (pro_b_gan_infer.py:97-98): the CUDA-backed modules use the oracle's key names."""
    import modular_prot_b_gan as m
    Go, Do = synth.make_models(oracle.ModularGenerator, oracle.ModularDiscriminator)
    G, D = m.ModularGenerator(128, 64), m.ModularDiscriminator(128, 1024)
    assert G.load_state_dict(Go.state_dict(), strict=True).missing_keys == []
    assert D.load_state_dict(Do.state_dict(), strict=True).missing_keys == []
    assert m.Generator is m.ModularGenerator and m.Discriminator is m.ModularDiscriminator


def test_batchnorm_fold_equals_eval_batchnorm(oracle, synth):
    """Load-time fold (legal in eval / no_grad, :106-107, :133) with NON-default running stats."""
    from pbg.engine import fold_linear_bn
    Go, _ = synth.make_models(oracle.ModularGenerator, oracle.ModularDiscriminator)
    lin, bn = Go.net[0], Go.net[1]
    assert not torch.allclose(bn.running_var, torch.ones_like(bn.running_var))
    x = torch.randn(64, lin.in_features, generator=torch.Generator().manual_seed(7))
    with torch.no_grad():
        want = bn(lin(x))
        W, b = fold_linear_bn(lin, bn)
        got = x @ W.T + b
    assert (got - want).abs().max().item() <= 2e-5
    W2, b2 = fold_linear_bn(Go.net[6], None)
    assert torch.equal(W2, Go.net[6].weight.detach()) and torch.equal(b2, Go.net[6].bias.detach())


def test_shard_bounds_cover_the_batch_exactly():
    from pbg import shard
    for B in (0, 1, 7, 16, 4096, 32768, 32771):
        for ws in (1, 2, 3, 4, 8):
            spans = [shard.shard_bounds(B, ws, r) for r in range(ws)]
            assert spans[0][0] == 0 and spans[-1][1] == B
            assert all(spans[i][1] == spans[i + 1][0] for i in range(ws - 1))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1 and sizes == shard.shard_sizes(B, ws)
    assert shard.shard_bounds(32768, 8, 3) == (3 * 4096, 4 * 4096)
    with pytest.raises(ValueError):
        shard.shard_bounds(8, 2, 2)


_GLOO_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path[:0] = [os.environ["PBG_PKG"], os.environ["PBG_ROOT"]]
from pbg import shard, synth
from oracle import prot_b_gan_oracle as oracle   # tests may use the oracle
rank, ws = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=ws)
torch.set_num_threads(1)
for B in (64, 37):   # even and ragged
    G, D = synth.make_models(oracle.ModularGenerator, oracle.ModularDiscriminator)
    node_emb, rel_w = synth.make_tables(num_entities=2048)
    trip, z = synth.make_triplets(B, num_entities=2048), synth.make_latents(B)
    with torch.no_grad():
        def run(tr, zz):
            h, r, t = node_emb[tr[:, 0]], rel_w[tr[:, 1]], node_emb[tr[:, 2]]
            return G(h, r, zz), D(h, r, t)
        full_g, full_d = run(trip, z)
        lo, hi = shard.shard_bounds(B, ws, rank)
        loc_g, loc_d = run(shard.take_shard(trip, ws, rank), shard.take_shard(z, ws, rank))
    got_g = shard.all_gather_rows(loc_g, B)
    got_d = shard.all_gather_rows(loc_d, B)
    assert got_g.shape == full_g.shape and got_d.shape == full_d.shape
    # row-wise map: sharding by batch index then all-gathering must reproduce the unsharded pass
    assert torch.allclose(got_g, full_g, atol=1e-6) and torch.allclose(got_d, full_d, atol=1e-6), (rank, B)
    assert torch.equal(got_g[lo:hi], loc_g)
dist.destroy_process_group()
print("OK", rank)
"""


def _free_port() -> int:
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_batch_sharding_plus_allgather_world_size_2_gloo(tmp_path):
    """The N > 1 path on CPU: 2 gloo ranks shard by batch index, run their shard, all-gather, compare with the
    unsharded pass."""
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER)
    port = _free_port()
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port),
                   PBG_PKG=str(ROOT / "pro-b-gan_b200"), PBG_ROOT=str(ROOT), OMP_NUM_THREADS="1")
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and f"OK {r}" in o, o


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", str(ROOT / "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_bench_reference_arm_prints_one_json_line(tmp_path):
    import json
    import numpy as np
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "3",
                          "--batch", "256", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "samples/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0
    # --dump-outputs: what the last timed step returned, float32, one row per triplet
    shapes = {"gen_out": (256, 128), "gen_scores": (256,), "logits": (256,), "probs": (256,)}
    assert sorted(p.name for p in tmp_path.iterdir()) == sorted(f"{k}.npy" for k in shapes)
    for k, shape in shapes.items():
        a = np.load(tmp_path / f"{k}.npy")
        assert a.dtype == np.float32 and a.shape == shape and np.isfinite(a).all(), k
    assert np.allclose(np.load(tmp_path / "probs.npy"), 1 / (1 + np.exp(-np.load(tmp_path / "logits.npy"))), atol=1e-6)


def test_bench_dump_outputs_keeps_a_seeded_sample_under_the_limit(tmp_path):
    import numpy as np
    bench = _bench_module()
    bench.DUMP_MAX_BYTES = 3000
    g = torch.Generator().manual_seed(5)
    arrays = {"gen_out": torch.randn(100, 8, generator=g), "logits": torch.randn(100, generator=g)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["gen_out.npy", "logits.npy", "rows.npy"]
    assert sum((tmp_path / "a" / f).stat().st_size for f in files) <= 3000
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert rows.dtype == np.float64 and 0 < len(rows) < 100 and (np.diff(rows) > 0).all()
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f   # the same sample every time
    assert np.array_equal(np.load(tmp_path / "a" / "gen_out.npy"), arrays["gen_out"].numpy()[rows.astype(int)])


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_bench_product_arm_has_no_cpu_fallback():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "1"], capture_output=True, text=True,
                         timeout=300)
    assert out.returncode != 0 and "no CPU fallback" in (out.stdout + out.stderr)


def test_bench_reference_arm_under_torchrun_prints_one_line_from_rank_0():
    """N > 1: the driver launches the reference arm like the product arm; rank 0 alone measures and prints."""
    import json
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), str(ROOT / "bench.py"), "--impl",
                          "reference", "--gpus", "2", "--steps", "2", "--warmup", "3", "--batch", "256"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["n_gpus"] == 2 and line["value"] > 0


def test_top_k_is_validated_on_the_host_before_anything_is_launched():
    """torch.topk's own error for k > rows (pro_b_gan_infer.py:151 raises RuntimeError), and this library's limit."""
    from pbg.engine import Engine
    Engine.validate_top_k(10, 65536)
    Engine.validate_top_k(512, 65536)
    with pytest.raises(RuntimeError, match="out of range"):
        Engine.validate_top_k(11, 10)
    with pytest.raises(RuntimeError):
        Engine.validate_top_k(0, 10)
    with pytest.raises(NotImplementedError, match="512"):
        Engine.validate_top_k(513, 65536)


def test_bench_flop_and_config_table_match_the_survey():
    """bench.py's algorithmic flop counts are SURVEY.md 8d's (2*K*N per Linear) for both BASELINE model shapes."""
    bench = _bench_module()
    assert bench.flops_per_sample(128, 64, 1024) == (3014656, 1836032)
    assert bench.flops_per_sample(256, 64, 4096) == (40370176, 23072768)
    assert bench.CONFIGS["base"]["batch"] == 4096 and bench.CONFIGS["wide"]["batch"] == 1024


def test_clock_sampler_summary_without_nvml_has_every_key():
    """bench.py's `clocks` entry: the sampler degrades to empty readings (never raises) where NVML has no device, and the
    keys the driver and DESIGN.md quote are always present."""
    from pbg.clocks import ClockSampler
    with ClockSampler(0, period_s=0.001) as clk:
        pass
    s = clk.summary()
    for key in ("sm_mhz", "sm_max_mhz", "reasons", "samples", "power_w", "power_w_max", "power_limit_w", "power_kind"):
        assert key in s
    assert isinstance(s["reasons"], list)


def test_traffic_record_names_a_figure_for_both_pass_forms():
    """profiles/traffic.json: bench.py's roofline.traffic follows the mode it runs (--stage-ahead 2 by default, 0 = fused
    gather); both figures and their provenance are recorded."""
    import json
    tj = json.loads((ROOT / "profiles" / "traffic.json").read_text())
    assert tj["pass_fused"] < tj["pass_stage2"] < 4 * 11.7e6       # algorithmic: 11.7 MB per 4096-triplet pass
    assert "dram_steady" in tj["source"]
