"""bench.py's JSON contract on the leg that runs without a GPU: `--impl reference` (the reference's CPU algorithm for the
path = the C++ oracle port) prints ONE JSON line with the keys the driver reads."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "ctxt_mults_per_s" and d["unit"] == "mult/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "mult/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("ckks_m2^17")


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_both_arms_describe_the_same_workload():
    """The driver compares the `config` dicts of the two arms: both come from bench.mult_config with the default batch."""
    sys.path.insert(0, ROOT)
    import importlib
    bench = importlib.import_module("bench")
    cfg = bench.mult_config(32)
    assert cfg["workload"].startswith("ckks_m2^17") and (cfg["l_in"], cfg["l"], cfg["K"], cfg["digits"]) == (20, 19, 10, 2)
    assert cfg["alg_bytes_per_mult"] == bench.ROW_BYTES * (4 * 20 + 2 * 2 * 29 + 2 * 19) == 122683392      # SURVEY 8d
    assert bench.alg_bytes_per_keyswitch(26, 9, 3) == bench.ROW_BYTES * 340                                   # config 3: 178.3 MB
    assert bench.alg_bytes_per_keyswitch(29, 15, 2) == bench.ROW_BYTES * 321                                  # config 4: 168.3 MB
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=900)
    assert json.loads(r.stdout.strip().splitlines()[-1])["config"] == cfg
    for cores in (1, 8, 16, 128, 192):
        w, per = bench.cpu_layout(cores)
        assert w >= 1 and per >= 1 and w * per <= max(cores, 1)


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(cuda_lib, tmp_path):
    """--dump-outputs: the files hold, bit for bit, what warm-up + --steps in-place multiplies of the seeded inputs leave in
    c0 and c1 (replayed here through the engine), on the documented column sample and within the size budget."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from helib_b200 import Chain, Engine
    B, warmup, steps = 2, 3, 2
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup), "--batch", str(B),
                        "--no-cpu", "--no-e2e", "--no-ks", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
    assert sorted(os.listdir(tmp_path)) == ["c0.npy", "c1.npy"]
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64 * 10**6

    w = bench.WORKLOAD
    ch = Chain(w["m"], w["p"], w["r"], w["bits"], w["c"], lib=cuda_lib)
    E = Engine(w["m"], ch.primes, None, ch.digits, ch.special, lib=cuda_lib)
    S_in, S, full = ch.ctxt, ch.ctxt[:-1], ch.ctxt + ch.special
    rng = np.random.Generator(np.random.Philox(bench.SEED))

    def rand_dense(idx):
        out = np.zeros((E.np, E.N), dtype=np.uint64)
        for i in idx:
            out[i] = rng.integers(0, ch.primes[i], size=E.N, dtype=np.uint64)
        return out

    EA = [E.poly(rand_dense(full), full) for _ in ch.digits]
    EB = [E.poly(rand_dense(full), full) for _ in ch.digits]
    ops = [[E.poly(rand_dense(S_in), S_in) for _ in range(4)] for _ in range(B)]
    A0, A1, B0, B1 = ([o[k] for o in ops] for k in range(4))
    for _ in range(warmup + steps):
        E.mul_relin_moddown(A0, A1, B0, B1, S_in, S, 1, EA, EB)
    cols = bench.dump_columns(E.N, B, len(S))
    for name, polys in (("c0", A0), ("c1", A1)):
        got = np.load(tmp_path / (name + ".npy"))
        assert got.dtype == np.float64 and got.shape == (B, len(S), len(cols), 2)
        want = np.stack([p.download(S)[S][:, cols] for p in polys])
        assert (((got[..., 0].astype(np.uint64) << np.uint64(32)) | got[..., 1].astype(np.uint64)) == want).all(), name
    del A0, A1, B0, B1, ops, EA, EB
    E.close()


def test_product_arm_refuses_to_run_without_a_gpu():
    """No CPU fallback anywhere on the product path: without a CUDA device bench.py's own arm and smoke() stop with an error
    instead of timing (or checking) something else."""
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is visible: the refusal path is not reachable")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "3", "--no-cpu"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode != 0 and r.stdout.strip() == "" and "no CUDA device" in (r.stderr + r.stdout)
    r = subprocess.run([sys.executable, "-c", "import __graft_entry__ as g; g.smoke()"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and "no CUDA device" in r.stderr
