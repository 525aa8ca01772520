#!/usr/bin/env python
"""bench.py -- Ctxt x Ctxt multiply (+ rescale, relinearise, mod-down) throughput on B200.

Workload (BASELINE.json configs[1], SURVEY.md section 8d "config 2"): CKKS m=2^17 (N=2^16),
bits=1190, c=2 -> 20 ctxt + 10 special 60-bit primes ("L~30").  One *step* = one batch of B (default 32)
independent ciphertext pairs through the hot path
    modDownToSet(20 -> 19 ctxt primes) of both operands  ->  tensorProduct  ->  reLinearize
    (breakIntoDigits, keySwitchDigits over 29 rows)  ->  modDownToSet (drop the 10 special primes)
with explicit prime sets and synthetic uniform residues (the path is data-oblivious).

JSON line (one, rank 0): value = whole-job multiplies/s with operands resident in HBM; e2e = the
same through the C ABI with pinned HOST buffers (H2D of the operands and D2H of the result inside
the timed region); roofline = dominant kernel vs the measured HBM peak; cpu_baseline = the C++
oracle (restated NTL-path HElib) on the host cores.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference] [--dump-outputs DIR]

--dump-outputs DIR writes, after the timed steps, the two result parts c0 and c1 the timed path left in HBM (rows of the
19 ctxt primes) as DIR/c0.npy and DIR/c1.npy: float64 arrays [batch][19][columns][2] holding each 60-bit residue as
(high 32 bits, low 32 bits), both exact in float64, over a fixed seeded sample of coefficient columns that keeps the
two files under 64 MB together.  The inputs depend only on the arguments, so two builds run with the same arguments
can be compared file for file.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = {"name": "ckks_m2^17_bits1190_c2", "m": 1 << 17, "p": -1, "r": 1, "bits": 1190, "c": 2}
SEED = 20260922 + 2  # SURVEY 8d: Philox, seed = 20260922 + config index
ROW_BYTES = (1 << 16) * 8
DUMP_BYTES = 63 * 10**6    # --dump-outputs: data of all files together (under 64 MB with the .npy headers)
DUMP_COLUMNS = 2048        # --dump-outputs: sampled coefficient columns per row (fewer when the batch is large)


def alg_bytes_per_mult(l_in, l, K, d):
    """SURVEY.md 8d: B_mul = 8N*[4*l_in + 2d(l+K) + 2l] (each input/evk/output row moved once)."""
    return ROW_BYTES * (4 * l_in + 2 * d * (l + K) + 2 * l)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm = sorted(float(r[1]) for r in rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        if sm:
            out["sm_mhz"] = sm[len(sm) // 2]
            out["sm_max_mhz"] = float(rows[0][2])
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            seen = set()
            for r in rows:
                for k, nm in enumerate(names):
                    if len(r) >= 9 and r[5 + k].strip().lower().startswith("active"):
                        seen.add(nm)
            out["reasons"] = sorted(seen)
            out["samples"] = len(sm)
        return out


def bind_near_gpu(gpu):
    """Run this rank on the CPU cores next to its GPU (sysfs local_cpulist of the GPU's PCI device) before the pinned host
    buffers are allocated, so first-touch places them on that NUMA node: with 8 ranks streaming 640 MiB per step each, staging
    buffers on the far socket put the inter-socket link in the H2D path.  Best effort; returns the core list or None."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(gpu), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().splitlines()[0].strip().lower()
        dom, rest = out.split(":", 1)
        path = f"/sys/bus/pci/devices/{dom[-4:]}:{rest}/local_cpulist"
        cpus = set()
        for part in open(path).read().strip().split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return sorted(cpus)
    except Exception:
        pass
    return None


def mult_config(B):
    """The workload both arms are run on (identical dict in `config` of the GPU arm and of --impl reference)."""
    l_in, l, K, d = 20, 19, 10, 2
    return {"workload": WORKLOAD["name"], "N": 1 << 16, "l_in": l_in, "l": l, "K": K, "digits": d, "batch_per_gpu": B,
            "sharding": "independent ciphertexts per rank, no data-path collective",
            "l2": f"inputs larger than L2 ({B * 4 * l_in * ROW_BYTES / 2**20:.0f} MiB of operands per step)",
            "operands": "updated in place: from step 2 on a step's inputs are the previous step's outputs (the path is data-oblivious)",
            "alg_bytes_per_mult": alg_bytes_per_mult(l_in, l, K, d)}


def dump_columns(N, B, l):
    """The coefficient columns --dump-outputs keeps: a sorted sample, fixed by SEED, sized so that two parts of B x l rows
    at 16 bytes per residue fit DUMP_BYTES."""
    import numpy as np
    n = max(1, min(N, DUMP_COLUMNS, DUMP_BYTES // (2 * B * l * 16)))
    return np.sort(np.random.Generator(np.random.Philox(SEED)).choice(N, size=n, replace=False))


def dump_outputs(path, parts, S, N):
    """Write each named list of result polys as path/<name>.npy (layout in the module docstring)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    cols = dump_columns(N, len(next(iter(parts.values()))), len(S))
    for name, polys in parts.items():
        res = np.stack([p.download(S)[S][:, cols] for p in polys])
        np.save(os.path.join(path, name + ".npy"), np.stack([res >> np.uint64(32), res & np.uint64(0xFFFFFFFF)], axis=-1).astype(np.float64))


def cpu_layout(cores):
    """Concurrent multiplies x threads per multiply: the reference threads one multiply across primes / coefficients
    (NTL_EXEC_RANGE, src/DoubleCRT.cpp:79-84), which cannot occupy a many-core host (<= 30 rows); independent
    ciphertexts on independent thread groups is how a caller fills the box."""
    per = 8 if cores >= 16 else max(1, cores)
    workers = max(1, cores // per)
    return workers, per


KS_WORKLOADS = {
    # BASELINE.json configs[2]: BGV m=2^17 p=257 bits=1500 c=3 -- reLinearize/key-switch batch of 1024 ctxts, 1xB200
    "cfg3": {"name": "bgv_m2^17_p257_bits1500_c3", "m": 1 << 17, "p": 257, "r": 1, "bits": 1500, "c": 3, "shape": (26, 9, 3)},
    # BASELINE.json configs[3]: CKKS N=2^16 L=44 -- prime-sharded key-switch at 1/2/4/8 GPUs over NVLink
    "cfg4": {"name": "ckks_m2^17_bits1700_c2", "m": 1 << 17, "p": -1, "r": 1, "bits": 1700, "c": 2, "shape": (29, 15, 2)},
}


def alg_bytes_per_keyswitch(l, K, d):
    """SURVEY.md 8d: B_ks = 8N*[3l + 2d(l+K) + 2l] (3-part in, evk, 2-part out incl. the mod-down)."""
    return ROW_BYTES * (3 * l + 2 * d * (l + K) + 2 * l)


def bench_keyswitch_block(args, np, torch, dist, local, rank, world, peak):
    """BASELINE config 3: `--ks-count` independent 3-part BGV ciphertexts (p = 257: the ptxtSpace correction of
    scaleDownToSet is active) resident in HBM; one step = reLinearize + modDownToSet of every one of them
    (hb_relinearize + hb_scale_down in groups of --ks-group).  Independent ciphertexts per rank, no collective."""
    from helib_b200 import Chain, Engine
    wl = KS_WORKLOADS["cfg3"]
    ch = Chain(wl["m"], wl["p"], wl["r"], wl["bits"], wl["c"])
    assert (len(ch.ctxt), len(ch.special), len(ch.digits)) == wl["shape"], "chain shape differs from SURVEY section 8"
    E = Engine(wl["m"], ch.primes, None, ch.digits, ch.special, device=local)
    N, npr = E.N, E.np
    S, full, nd, p = ch.ctxt, ch.ctxt + ch.special, len(ch.digits), ch.p ** ch.r
    Sp = sorted(S + ch.special)
    rng = np.random.Generator(np.random.Philox(20260922 + 3 + 1000 * rank))

    def rand_dense(idx):
        out = np.zeros((npr, N), dtype=np.uint64)
        for i in idx:
            out[i] = rng.integers(0, ch.primes[i], size=N, dtype=np.uint64)
        return out

    EA = [E.poly(rand_dense(full), full) for _ in range(nd)]
    EB = [E.poly(rand_dense(full), full) for _ in range(nd)]
    count, grp = args.ks_count, min(args.ks_group, args.ks_count)
    nuniq = min(8, count)
    C = [[E.poly(rand_dense(S), S) if b < nuniq else E.poly() for _ in range(3)] for b in range(count)]
    for b0 in range(nuniq, count, nuniq):     # the remaining ciphertexts are device-side copies of the unique ones
        nb = min(nuniq, count - b0)
        for k in range(3):
            E.pointwise("copy", [C[b0 + j][k] for j in range(nb)], [C[j][k] for j in range(nb)], S)
    groups = [([c[0] for c in C[g:g + grp]], [c[1] for c in C[g:g + grp]], [c[2] for c in C[g:g + grp]]) for g in range(0, count, grp)]

    def step():
        for c0, c1, c2 in groups:
            E.relinearize(c0, c1, c2, S, EA, EB)
            E.scale_down(c0 + c1, Sp, S, p)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    steps = max(1, min(args.steps, args.ks_steps))
    for _ in range(3):
        step()
    E.reset_stats()
    barrier()
    E.mark_begin()
    for _ in range(steps):
        step()
    ms = E.mark_end()
    barrier()
    st = E.stats()
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    E.profile(True)
    c0, c1, c2 = groups[0]
    E.relinearize(c0, c1, c2, S, EA, EB)
    E.scale_down(c0 + c1, Sp, S, p)
    E.profile(False)
    prof = sorted(E.profile_results(), key=lambda r: -r["ms"])
    tot = sum(r["ms"] for r in prof) or 1.0
    l, K = len(S), len(ch.special)
    bks = alg_bytes_per_keyswitch(l, K, nd)
    v = world * count * steps / (ms / 1000.0)
    top = prof[0] if prof else None
    out = {
        "metric": "key_switches_per_s", "value": v, "unit": "keyswitch/s", "steps": steps, "warmup": 3, "ms_per_step": ms / steps,
        "config": {"workload": wl["name"], "N": N, "l": l, "K": K, "digits": nd, "ptxt_space": p, "ciphertexts_per_gpu": count, "group": grp,
                   "resident_bytes": count * 3 * l * ROW_BYTES, "alg_bytes_per_keyswitch": bks, "alg_bytes_per_keyswitch_without_evk": bks - 2 * nd * (l + K) * ROW_BYTES,
                   "sharding": "independent ciphertexts per rank, no data-path collective"},
        "alg_roofline": {"achieved_GBps": v / world * bks / 1e9, "peak_GBps": peak, "frac": v / world * bks / 1e9 / peak},
        "roofline": None if top is None else {"bound": "hbm", "kernel": top["kernel"], "achieved": top["bytes"] / (top["ms"] / 1000.0) / 1e9, "peak": peak, "unit": "GB/s",
                                             "frac": top["bytes"] / (top["ms"] / 1000.0) / 1e9 / peak, "share_of_step": top["ms"] / tot, "traffic": None},
        "gpu_launches": st["launches"], "exact_crt_fallbacks": st["exact_fallbacks"],
        "kernels": [{"kernel": r["kernel"], "launches": r["launches"], "ms": round(r["ms"], 4), "share": round(r["ms"] / tot, 4)} for r in prof],
    }
    del groups, C, EA, EB, c0, c1, c2
    import gc
    gc.collect()          # polys are freed by their finalisers (before the context goes away)
    E.close()
    return out


def bench_general_m_block(np, torch, local):
    """BASELINE config 5's ring (m = 21845, phi(m) = 16384, Bluestein rows of length 2^16; p=2, bits=580, c=2 as
    tests/GTestThinBootstrapping.cpp:102, bootstrappable chain): row transforms/s, relinearise + mod-down/s and hoisted
    rotations/s of the DoubleCRT layer underneath recryption (the linear maps and digit extraction of thinReCrypt are callers
    above the boundary).  Rank 0 only."""
    from helib_b200 import Chain, Engine
    m, p, r, bits, c = 21845, 2, 1, 580, 2
    ch = Chain(m, p, r, bits, c, bootstrappable=True)
    E = Engine(m, ch.primes, None, ch.digits, ch.special, device=local)
    N, npr = E.N, E.np
    S, full = ch.ctxt, ch.ctxt + ch.special
    Sp = sorted(full)
    nd = len(ch.digits)
    rng = np.random.Generator(np.random.Philox(20260922 + 5))
    B = 8

    def rand(idx):
        out = np.zeros((npr, N), dtype=np.uint64)
        for i in idx:
            out[i] = rng.integers(0, ch.primes[i], size=N, dtype=np.uint64)
        return out

    EA = [E.poly(rand(full), full) for _ in range(nd)]
    EB = [E.poly(rand(full), full) for _ in range(nd)]
    C = [[E.poly(rand(S), S) for _ in range(3)] for _ in range(B)]
    C0, C1, C2 = ([x[k] for x in C] for k in range(3))
    O0, O1 = [E.poly() for _ in range(B)], [E.poly() for _ in range(B)]

    def timed(fn, steps):
        for _ in range(2):
            fn()
        E.sync()
        E.mark_begin()
        for _ in range(steps):
            fn()
        return E.mark_end() / steps

    t_f = timed(lambda: E.ntt_fwd(C0, S), 5)
    t_i = timed(lambda: E.ntt_inv(C0, S), 5)

    def ks():
        E.relinearize(C0, C1, C2, S, EA, EB)
        E.scale_down(C0 + C1, Sp, S, p)
    t_ks = timed(ks, 3)
    digs = E.break_into_digits(C1, S)
    k = next(t for t in range(2, m) if np.gcd(t, m) == 1)
    t_rot = timed(lambda: E.automorph_keyswitch_digits(digs, S, C0, k, EA, EB, O0, O1), 3)
    rows = B * len(S)
    out = {"workload": "bgv_m21845_p2_bits580_c2_bootstrappable", "m": m, "phim": N, "bluestein_length": 65536, "division_length": 1 << (max(N, 2 * (m - N) - 1) - 1).bit_length(), "e": ch.e_param, "e_prime": ch.e_prime_param,
           "primes": {"ctxt": len(S), "special": len(ch.special), "digits": nd}, "batch": B,
           "fwd_rows_per_s": rows / (t_f / 1e3), "inv_rows_per_s": rows / (t_i / 1e3),
           "relin_moddown_per_s": B / (t_ks / 1e3), "hoisted_rotations_per_s": B / (t_rot / 1e3),
           "ms": {"fwd": t_f, "inv": t_i, "relin_moddown": t_ks, "hoisted_rotation": t_rot}}
    del EA, EB, C, C0, C1, C2, O0, O1, digs
    return out


def bench_sharded_block(args, np, torch, dist, local, rank, world, peak):
    """BASELINE config 4: ONE stream of ciphertexts, every ciphertext's rows sharded by RNS prime index over the ranks
    (helib_b200/sharded.py): key-switches/s (strong scaling), exchange bytes, and a bit-exact check of the rows each rank
    owns against the unsharded engine path run on the same inputs inside this process."""
    from helib_b200 import Chain, Engine
    from helib_b200.sharded import ShardedKeySwitch
    wl = KS_WORKLOADS["cfg4"]
    ch = Chain(wl["m"], wl["p"], wl["r"], wl["bits"], wl["c"])
    assert (len(ch.ctxt), len(ch.special), len(ch.digits)) == wl["shape"], "chain shape differs from SURVEY section 8"
    E = Engine(wl["m"], ch.primes, None, ch.digits, ch.special, device=local)
    side = torch.cuda.Stream()            # engine kernels, torch index ops and NCCL all run ordered on this stream
    prev = torch.cuda.current_stream()
    torch.cuda.set_stream(side)
    E.set_stream(side.cuda_stream)
    N, npr, B = E.N, E.np, args.sharded_batch
    S, full, nd = ch.ctxt, ch.ctxt + ch.special, len(ch.digits)
    rng = np.random.Generator(np.random.Philox(20260922 + 4))      # the same data on every rank

    def rand_dense(idx):
        out = np.zeros((npr, N), dtype=np.uint64)
        for i in idx:
            out[i] = rng.integers(0, ch.primes[i], size=N, dtype=np.uint64)
        return out

    evk = [rand_dense(full) for _ in range(2 * nd)]
    nuniq = min(4, B)
    cts = [[rand_dense(S) for _ in range(3)] for _ in range(nuniq)]
    res = {}
    # modes: (name, peer stores?, ranks per prime-sharded group).  Pure sharding = one group over all ranks (strong scaling of ONE
    # stream of B ciphertexts per step); with >= 4 ranks also independent groups of 4 / 2 ranks side by side, each sharding its own
    # stream by prime index (the conversion kernel needs all source rows of a column on chip but has only (l+K)/R target rows of
    # work for them, so small groups use the SMs better -- DESIGN.md section 6).
    modes = [("local", False, 1)] if world == 1 else [("p2p", True, world), ("gather", False, world)]
    if world > 1:
        modes += [(f"p2p_groups_of_{g}", True, g) for g in (4, 2) if world > g and world % g == 0]
    subgroups = {}
    for _, _, g in modes:
        if 1 < g < world and g not in subgroups:
            gl = [dist.new_group(list(range(i, i + g))) for i in range(0, world, g)]   # every rank creates every group, same order
            subgroups[g] = gl[rank // g]
    for mode, use_p2p, gsz in modes:
        ngroups = world // gsz
        grp = subgroups.get(gsz)
        KS = ShardedKeySwitch(E, ch.ctxt, ch.special, ch.digits, rank=rank % gsz, world=gsz, device=f"cuda:{local}", p2p=use_p2p, group=grp)
        own_full, oS = KS.owned(full), KS.owned(S)
        EA = [E.poly(evk[i], own_full) for i in range(nd)]
        EB = [E.poly(evk[nd + i], own_full) for i in range(nd)]
        C = [[E.poly(cts[b % nuniq][k], oS) for k in range(3)] for b in range(B)]
        digs = [[E.poly() for _ in range(nd)] for _ in range(B)]
        C0, C1, C2 = ([c[k] for c in C] for k in range(3))

        def step():
            Sp_ = KS.relinearize(C0, C1, C2, S, EA, EB, digs)
            KS.mod_down(C0 + C1, Sp_, S, 1)

        def barrier():
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        # ---- parity inside the run: rows this rank owns == the unsharded engine path on the same inputs
        step()
        torch.cuda.synchronize()
        got = [(C0[b].download(oS), C1[b].download(oS)) for b in range(nuniq)]
        FA = [E.poly(evk[i], full) for i in range(nd)]
        FB = [E.poly(evk[nd + i], full) for i in range(nd)]
        ok = True
        for b in range(nuniq):
            f0, f1, f2 = (E.poly(cts[b][k], S) for k in range(3))
            E.relinearize([f0], [f1], [f2], S, FA, FB)
            E.scale_down([f0, f1], sorted(S + ch.special), S, 1)
            r0, r1 = f0.download(oS), f1.download(oS)
            ok = ok and bool((got[b][0][oS] == r0[oS]).all() and (got[b][1][oS] == r1[oS]).all())
        del FA, FB
        if world > 1:
            t = torch.tensor([1 if ok else 0], device="cuda", dtype=torch.int32)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            ok = bool(t.item())
        for _ in range(3):
            step()
        E.reset_stats()
        step()
        launches_per_step = E.stats()["launches"]
        barrier()
        run, graphed = step, False
        try:     # ~30 launches + the exchange steps per pass: replay them as one CUDA graph
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                step()
            run, graphed = g.replay, True
            for _ in range(2):
                run()
        except Exception as ex:
            if rank == 0:
                print(f"[bench] sharded key switch: CUDA graph capture failed ({type(ex).__name__}: {ex}); running eagerly", file=sys.stderr)
        barrier()
        steps = max(1, min(args.steps, args.ks_steps * 4))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            run()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        E.profile(True)
        step()
        E.profile(False)
        prof = sorted(E.profile_results(), key=lambda r: -r["ms"])
        l, K = len(S), len(ch.special)
        bks = alg_bytes_per_keyswitch(l, K, nd)
        v = ngroups * B * steps / (ms / 1000.0)
        res[mode] = {
            "value": v, "unit": "keyswitch/s", "ms_per_step": ms / steps, "steps": steps, "cuda_graph": graphed, "bit_exact_vs_unsharded": ok,
            "ranks_per_group": gsz, "groups": ngroups, "ciphertexts_per_step": ngroups * B,
            "gpu_launches_per_step": launches_per_step,
            "exchange_bytes_per_keyswitch": (l + 2 * K) * ROW_BYTES if gsz > 1 else 0, "exchanges_per_step": (nd + 1) if gsz > 1 else 0,
            "alg_roofline_frac": v * bks / 1e9 / (peak * world),
            "phase_ms": [{"kernel": r["kernel"], "launches": r["launches"], "ms": round(r["ms"], 4)} for r in prof],
            "engine_kernel_ms_per_step": round(sum(r["ms"] for r in prof), 4),
        }
        del C, digs, EA, EB, KS
    torch.cuda.set_stream(prev)
    pure = [r for r in res.values() if r["groups"] == 1]
    best = max(pure, key=lambda r: r["value"])                      # the headline of this block: ONE group over all ranks
    hybrid = max(res.values(), key=lambda r: r["value"])
    l, K = len(S), len(ch.special)
    out = {"metric": "key_switches_per_s", "value": best["value"], "unit": "keyswitch/s", "scaling": "strong", "n_gpus": world,
           "best_grouping": {"ranks_per_group": hybrid["ranks_per_group"], "groups": hybrid["groups"], "value": hybrid["value"],
                             "note": "independent prime-sharded groups side by side (one stream of ciphertexts per group)"},
           "config": {"workload": wl["name"], "N": N, "l": l, "K": K, "digits": nd, "batch": B, "sharding": "rows by RNS prime index, round-robin within ctxt / special primes; evk sharded identically",
                      "alg_bytes_per_keyswitch": alg_bytes_per_keyswitch(l, K, nd)},
           "bit_exact_vs_unsharded": all(r["bit_exact_vs_unsharded"] for r in res.values()), "modes": res}
    return out


def oracle_setup(nthreads):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import orc
    import pyoracle as po
    w = WORKLOAD
    ch = po.build_mod_chain(w["m"], w["p"], w["r"], w["bits"], w["c"])
    psis = [po.find_psi(q, ch.m) for q in ch.primes]
    O = orc.Oracle(ch.phim, ch.m, ch.primes, psis, ch.digits, ch.special, nthreads=nthreads)
    rng = np.random.Generator(np.random.Philox(SEED))
    full = ch.ctxt + ch.special
    nd = len(ch.digits)
    evk_a = np.stack([O.random(rng, full) for _ in range(nd)])
    evk_b = np.stack([O.random(rng, full) for _ in range(nd)])
    ops = [O.random(rng, ch.ctxt) for _ in range(4)]
    return ch, O, evk_a, evk_b, ops


def oracle_one_mult(ch, O, evk_a, evk_b, ops):
    """Host orchestration of Ctxt::multLowLvl + reLinearize + modDownToSet with explicit prime sets
    (reference: src/Ctxt.cpp:393-562,720-786,1681-1774) over the C++ oracle."""
    S_in, S = ch.ctxt, ch.ctxt[:-1]
    Sp = sorted(S + ch.special)
    parts = [x.copy() for x in ops]
    for x in parts:
        O.scale_down(x, S_in, S, 1)
    t0, t1, t2 = O.tensor(*parts, S)
    r0, r1 = O.relinearize(t0, t1, t2, S, evk_a, evk_b)
    O.scale_down(r0, Sp, S, 1)
    O.scale_down(r1, Sp, S, 1)
    return r0, r1


def time_oracle(steps, warmup, cores):
    """`steps` rounds of `workers` concurrent multiplies (one oracle context and thread group each; ctypes releases the GIL).
    Returns (multiplies/s, seconds, multiplies timed, workers, threads per multiply)."""
    import threading
    workers, per = cpu_layout(cores)
    ch, O, evk_a, evk_b, ops = oracle_setup(per)
    import orc
    Os = [O] + [orc.Oracle(ch.phim, ch.m, O.primes, O.psis, ch.digits, ch.special, nthreads=per) for _ in range(workers - 1)]

    def round_():
        th = [threading.Thread(target=oracle_one_mult, args=(ch, o, evk_a, evk_b, ops)) for o in Os[1:]]
        for t_ in th:
            t_.start()
        oracle_one_mult(ch, Os[0], evk_a, evk_b, ops)
        for t_ in th:
            t_.join()

    for _ in range(warmup):
        round_()
    t = time.perf_counter()
    for _ in range(steps):
        round_()
    dt = time.perf_counter() - t
    return steps * workers / dt, dt, steps * workers, workers, per


def run_reference(args):
    """--impl reference: the reference's CPU algorithm for this path (the C++ oracle: HElib itself
    cannot be built here, DESIGN.md section 5) on all host cores; each step = 1 multiply."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    v, dt, nmul, workers, per = time_oracle(args.steps, min(args.warmup, 1), cores)
    line = {
        "impl": "reference", "metric": "ctxt_mults_per_s", "value": v, "unit": "mult/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": mult_config(args.batch),
        "cpu_baseline": {"value": v, "unit": "mult/s", "cores": workers * per, "kind": "port",
                         "sample": f"each step = {workers} concurrent multiplies of the batch (bounded sample), {per} threads per multiply across primes/coefficients; "
                                   f"{nmul} multiplies in {dt:.1f}s; C++ oracle restating NTL-path HElib (HElib itself is unbuildable here: NTL/GMP absent)"},
        "e2e": {"value": v, "unit": "mult/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=32, help="independent ciphertext pairs per step and GPU")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=48, help="multiplies timed for cpu_baseline")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-streams", type=int, default=4, help="engine contexts (CUDA streams) the e2e loop spreads the batch over")
    ap.add_argument("--no-ks", action="store_true", help="skip the key-switch blocks (BASELINE configs 3 and 4)")
    ap.add_argument("--ks-count", type=int, default=1024, help="config 3: ciphertexts resident per GPU (one step switches all of them)")
    ap.add_argument("--ks-group", type=int, default=64, help="config 3: ciphertexts per hb_relinearize / hb_scale_down call")
    ap.add_argument("--ks-steps", type=int, default=3, help="config 3: timed passes over the resident ciphertexts (at most --steps)")
    ap.add_argument("--sharded-batch", type=int, default=32, help="config 4: ciphertexts per step of the prime-sharded key switch")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the results of the last one as DIR/c0.npy, DIR/c1.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    if args.warmup < 3:
        args.warmup = 3

    import numpy as np
    import torch
    from helib_b200 import Chain, Engine

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    all_cpus = os.sched_getaffinity(0)
    near = bind_near_gpu(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    w = WORKLOAD
    ch = Chain(w["m"], w["p"], w["r"], w["bits"], w["c"])
    assert (len(ch.ctxt), len(ch.special), len(ch.digits)) == (20, 10, 2), "chain shape differs from SURVEY section 8"
    E = Engine(w["m"], ch.primes, None, ch.digits, ch.special, device=local)
    N, npr = E.N, E.np
    S_in, S = ch.ctxt, ch.ctxt[:-1]
    full = ch.ctxt + ch.special
    nd = len(ch.digits)
    B = args.batch
    rng = np.random.Generator(np.random.Philox(SEED + 1000 * rank))

    def rand_dense(idx):
        out = np.zeros((npr, N), dtype=np.uint64)
        for i in idx:
            out[i] = rng.integers(0, ch.primes[i], size=N, dtype=np.uint64)
        return out

    EA = [E.poly(rand_dense(full), full) for _ in range(nd)]
    EB = [E.poly(rand_dense(full), full) for _ in range(nd)]
    # pinned host staging (torch is plumbing for pinned memory only)
    host_in = torch.empty((B, 4, npr, N), dtype=torch.int64, pin_memory=True)
    host_out = torch.empty((B, 2, npr, N), dtype=torch.int64, pin_memory=True)
    hin = host_in.numpy().view(np.uint64)
    for b in range(B):
        for k in range(4):
            hin[b, k] = rand_dense(S_in)
    polys = [[E.poly() for _ in range(4)] for _ in range(B)]

    def upload_all():
        for b in range(B):
            for k in range(4):
                polys[b][k].upload_ptr(host_in[b, k].data_ptr(), S_in)

    def download_all():
        for b in range(B):
            for k in range(2):
                polys[b][k].download_async_ptr(host_out[b, k].data_ptr(), S)

    A0, A1, B0, B1 = ([polys[b][k] for b in range(B)] for k in range(4))

    def step():
        E.mul_relin_moddown(A0, A1, B0, B1, S_in, S, 1, EA, EB)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    upload_all()
    E.sync()
    sampler = ClockSampler(local) if rank == 0 else None   # nvidia-smi needs ~0.2 s to deliver its first sample
    for _ in range(args.warmup):
        step()
    E.reset_stats()
    barrier()
    E.mark_begin()
    for _ in range(args.steps):
        step()
    ms = E.mark_end()
    barrier()
    st = E.stats()
    launches = st["launches"]
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = world * B * args.steps / (ms / 1000.0)
    if args.dump_outputs and rank == 0:     # before the e2e loop, which reuses these polys
        dump_outputs(args.dump_outputs, {"c0": A0, "c1": A1}, S, N)

    # ---- e2e: host buffers -> H2D -> hot path -> D2H, every step.  Two engine contexts (two CUDA
    #      streams), each with half of the batch, so the PCIe copies of one half overlap the kernels of
    #      the other -- the way a caller keeps the link busy; same pinned host buffers, same results.
    e2e = None
    if not args.no_e2e:
        ns = max(1, min(args.e2e_streams, B))
        engines = [E] + [Engine(w["m"], ch.primes, None, ch.digits, ch.special, device=local) for _ in range(ns - 1)]
        halves = [(engines[k], list(range(k * B // ns, (k + 1) * B // ns))) for k in range(ns)]
        ctxs = []
        for eng, items in halves:
            if eng is E:
                ea, eb, pl = EA, EB, [polys[b] for b in items]
            else:
                ea = [eng.poly() for _ in range(nd)]
                eb = [eng.poly() for _ in range(nd)]
                tmp = np.zeros((npr, N), dtype=np.uint64)
                for src, dst in list(zip(EA, ea)) + list(zip(EB, eb)):
                    src.download(full, tmp)
                    dst.upload(tmp, full)
                pl = [[eng.poly() for _ in range(4)] for _ in items]
            ctxs.append((eng, items, ea, eb, pl))

        def e2e_step():
            for eng, items, ea, eb, pl in ctxs:
                for j, b in enumerate(items):
                    for k in range(4):
                        pl[j][k].upload_ptr(host_in[b, k].data_ptr(), S_in)
                eng.mul_relin_moddown([p_[0] for p_ in pl], [p_[1] for p_ in pl], [p_[2] for p_ in pl], [p_[3] for p_ in pl], S_in, S, 1, ea, eb)
                for j, b in enumerate(items):
                    for k in range(2):
                        pl[j][k].download_async_ptr(host_out[b, k].data_ptr(), S)

        for _ in range(2):
            e2e_step()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step()
        for eng, *_ in ctxs:
            eng.sync()
        ems = (time.perf_counter() - t0) * 1000.0   # host clock around fully synchronised work on both streams
        barrier()
        if world > 1:
            t = torch.tensor([ems], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ems = float(t.item())
        e2e = {"value": world * B * args.steps / (ems / 1000.0), "unit": "mult/s",
               "h2d_bytes_per_step": B * 4 * len(S_in) * ROW_BYTES, "d2h_bytes_per_step": B * 2 * len(S) * ROW_BYTES,
               "ms_per_step": ems / args.steps, "streams": len(ctxs), "timing": "host perf_counter around synchronised streams",
               "host_cores_near_gpu": len(near) if near else None}

    clocks = sampler.stop() if sampler else {}   # sampled from warm-up through the timed region and the e2e loop
    # ---- per-kernel profile (one extra step bracketed by events per launch) -> roofline
    peak, peak_kind = peaks()
    E.profile(True)
    step()
    E.profile(False)
    prof = sorted(E.profile_results(), key=lambda r: -r["ms"])
    tot_ms = sum(r["ms"] for r in prof) or 1.0
    roof = None
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except Exception:
        tj = {}
    if prof:
        top = prof[0]
        base = top["kernel"].replace("_subscale", "")
        if base in tj:
            t8 = tj[base].get("avg_dram_bytes_per_launch_at_batch8")
            if t8:
                traffic = t8 * B / 8.0                  # older capture at batch 8; DRAM bytes per launch scale with the items per launch
            elif tj[base].get("avg_dram_bytes_per_launch"):
                traffic = tj[base]["avg_dram_bytes_per_launch"] * B / float(tj[base].get("batch") or B)
        ach = top["bytes"] / (top["ms"] / 1000.0) / 1e9
        roof = {"bound": "hbm", "kernel": top["kernel"], "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "peak_kind": peak_kind, "binding_unit": "integer pipes (ncu: FMA-heavy 67-72 %, ALU 41 % in k1_conv; DRAM 6 %) -- see profiles/", "traffic": traffic, "traffic_source": ("profiles/ncu_traffic.json: " + str(tj.get("source", ""))[:160]) if traffic else None, "share_of_step": top["ms"] / tot_ms,
                "launches_per_step": top["launches"], "avg_launch_ms": top["ms"] / top["launches"],
                "alg_bytes_per_launch": top["bytes"] / top["launches"]}
    kernels = [{"kernel": r["kernel"], "launches": r["launches"], "ms": round(r["ms"], 4), "share": round(r["ms"] / tot_ms, 4),
                "alg_GBps": round(r["bytes"] / (r["ms"] / 1000.0) / 1e9, 1) if r["ms"] > 0 else None} for r in prof]

    l_in, l, K, d = len(S_in), len(S), len(ch.special), nd
    st_mult = st
    # ---- the key-switch blocks (BASELINE configs 3 and 4); every rank takes part.  The multiply block's ~8 GB stay allocated.
    ks = sharded = None
    if not args.no_ks:
        import gc
        gc.collect()
        ks = bench_keyswitch_block(args, np, torch, dist if world > 1 else None, local, rank, world, peak)
        gc.collect()
        sharded = bench_sharded_block(args, np, torch, dist if world > 1 else None, local, rank, world, peak)
    if rank != 0:
        return _leave(world)
    general_m = None
    if not args.no_ks:
        try:
            general_m = bench_general_m_block(np, torch, local)
        except Exception as ex:   # a secondary block must not take the headline line down
            general_m = {"error": f"{type(ex).__name__}: {ex}"}
    st = st_mult
    bmul = alg_bytes_per_mult(l_in, l, K, d)
    try:
        os.sched_setaffinity(0, all_cpus)     # the CPU baseline uses every host core
    except Exception:
        pass
    cpu = None
    if not args.no_cpu and world == 1:
        cores = os.cpu_count() or 1
        workers, per = cpu_layout(cores)
        v, dt, nmul, workers, per = time_oracle(max(1, args.cpu_sample // workers), 1, cores)
        cpu = {"value": v, "unit": "mult/s", "cores": workers * per, "kind": "port",
               "sample": f"{nmul} multiplies of the same workload ({workers} concurrent x {per} threads each), C++ oracle restating NTL-path HElib, {dt:.1f}s"}
    line = {
        "metric": "ctxt_mults_per_s", "value": value, "unit": "mult/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic",
        "config": mult_config(B),
        "alg_roofline": {"achieved_GBps": value / world * bmul / 1e9, "peak_GBps": peak, "frac": value / world * bmul / 1e9 / peak, "peak_kind": peak_kind},
        "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "kernels": kernels,
        "exact_crt_fallbacks": st["exact_fallbacks"],
        "keyswitch": ks, "sharded_keyswitch": sharded, "general_m": general_m,
    }
    print(json.dumps(line))
    _leave(world)


def _leave(world):
    """Leave without tearing NCCL down: destroy_process_group() after a captured graph that contains collectives can block
    for minutes; the results are already printed."""
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        import torch
        torch.cuda.synchronize()
        os._exit(0)


if __name__ == "__main__":
    main()
