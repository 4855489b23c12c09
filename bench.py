#!/usr/bin/env python3
"""bench.py -- hifi F-16 aircraft-steps/s of the fused Euler step on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this framework (CUDA, libf16_b200.so)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU code on the host cores

One bench "step" = one pass of the hot path over one batch: `--aircraft` aircraft (default 2^20, BASELINE cfg 2:
random +-5 % perturbations about the 10000 ft / 700 ft/s trim, hifi, xcg 0.25) advanced `--euler-steps` fused
explicit-Euler steps (default 10000 = 10 s of flight) by ONE launch of step_kernel.  For N > 1 (torchrun, one rank
per GPU) every rank owns its own 2^20 aircraft: aircraft never interact, so there is no data-path collective and
the scaling is weak; NCCL is used for the barrier, the max-over-ranks time and the gather of survivor statistics.

Printed JSON keys beyond the base contract:
  roofline      FP64-pipe roofline of step_kernel: achieved = aircraft-steps/s/GPU x 750 algorithmic flop
                (SURVEY.md 8d) vs the DFMA rate measured live on this GPU (f16_measure_fp64_peak); the HBM view of
                the same launch (320 B per aircraft per launch) is under "hbm".
  e2e           same metric through the host-buffer C ABI call step_batch(): pinned host arrays in, H2D + kernel +
                D2H inside the timed region.
  cpu_baseline  the reference's Nlplant/atmos (oracle/_ref/*.so, built from the reference sources) driven by the
                restated env.py step on the host cores, OpenMP over aircraft, on a bounded sample.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
sys.dont_write_bytecode = True   # the benchmark leaves the tree it runs from as it found it (no __pycache__)

FLOP_PER_STEP = {"open": 750.0, "lqr": 815.0}   # algorithmic FP64 flop per hifi aircraft-step (SURVEY.md 8d)
BYTES_PER_AIRCRAFT_LAUNCH = 320.0               # read 18 + 4, write 18 doubles, independent of K
# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the step kernel at the default workload (2^20 aircraft,
# K = 10000), from the ncu capture of this build (profiles/r02_step_hifi_fast_chunked_k10000_ncu_summary.md; the earlier captures
# are in profiles/r02_step_dram_traffic.md): 197.3 MB read + 116.8 MB written against
# 335.5 MB algorithmic (320 B x 2^20) + 4 MB of status words -- part of the state still sits in L2 from the copy that precedes
# the launch.  The time-chunked schedule (f16_step_fast.cu) passes the state through global memory between its 16 chunks of 625
# steps; its item order keeps a block of groups inside L2 from one chunk to the next (L2 hit rate 77 %), so that traffic never
# reaches DRAM (the first version of the schedule moved 5.4 GB per launch).  Reported only when the run is that workload.
NCU_DRAM_BYTES_PER_LAUNCH = {(1 << 20, "open", "fast"): 197_272_576 + 116_838_656}

# trim of the reference at 10000 ft / 700 ft/s, xcg 0.25, hifi (tests/golden/env_xcg25.npz, env.py:198-292)
GOLDEN = os.path.join(REPO, "tests", "golden")


def trim_state(tag):
    g = np.load(os.path.join(GOLDEN, f"env_{tag}.npz"))
    return g["x_trim"].copy(), g["u_trim"].copy(), list(g["mpc_x_idx"])


def perturbed_trim(n, x_trim, u_trim, seed, frac=0.05):
    """x_i = x_trim (1 + frac U(-1,1)); zero-valued trim entries get additive frac U(-1,1) (SURVEY.md 8d cfg 2)."""
    r = np.random.default_rng(seed)
    rx = r.uniform(-1, 1, (18, n))
    ru = r.uniform(-1, 1, (4, n))
    xt = x_trim[:, None]
    x = np.where(xt != 0, xt * (1 + frac * rx), frac * rx)
    x[0:2] = 0.0
    u = u_trim[:, None] * (1 + frac * ru)
    return np.ascontiguousarray(x), np.ascontiguousarray(u)


DUMP_AIRCRAFT = 1 << 17   # aircraft kept by --dump-outputs over all ranks: 19 doubles each, 20 MB in all


def dump_outputs(out_dir, x, status, rank=0, world=1):
    """--dump-outputs: what the last timed step returned, the state [18][n] as DIR/x.npy and the status words [n] as
    DIR/status.npy (float64, exact for the int32 bit masks); under several ranks every rank writes its own batch as
    DIR/x.rank<k>.npy and DIR/status.rank<k>.npy.  A batch above its share of DUMP_AIRCRAFT keeps a fixed seeded sample of
    aircraft in ascending order, the same columns in every run, so that two builds compare entry for entry."""
    n, keep = x.shape[1], DUMP_AIRCRAFT // world
    idx = np.arange(n) if n <= keep else np.sort(np.random.default_rng(0xD0).choice(n, keep, replace=False))
    sfx = f".rank{rank}" if world > 1 else ""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"x{sfx}.npy"), np.ascontiguousarray(x[:, idx], dtype=np.float64))
    np.save(os.path.join(out_dir, f"status{sfx}.npy"), status[idx].astype(np.float64))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


def dist_setup(n_gpus):
    """torch.distributed over NCCL when launched by torchrun; plain single process otherwise."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1:
        return None, 0, 1, local
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return dist, rank, world, local


# ---------------------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation on the host cores
# ---------------------------------------------------------------------------------------------------------------
def cpu_reference_rate(aircraft, euler_steps, seed, repeats=1, lqr=None):
    """aircraft-steps/s of the reference Nlplant/atmos under the restated env.py step, OpenMP over aircraft."""
    from oracle import PORT, REF, get_oracle
    o = get_oracle()
    o.set_threads(len(os.sched_getaffinity(0)))   # all host cores of this process, whatever OMP_NUM_THREADS says
    kind, be = ("reference", REF) if o.open_ref() else ("port", PORT)
    x_trim, u_trim, _ = trim_state("xcg25")
    x, u = perturbed_trim(aircraft, x_trim, u_trim, seed)
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        xf, st = o.step_batch(x, u, euler_steps, 0.001, 1, 0.25, lqr, be)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return aircraft * euler_steps / best, kind, o.max_threads(), float((st == 0).mean()), best, xf, st


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    aircraft, esteps = args.ref_aircraft, args.ref_euler_steps
    for _ in range(args.warmup):
        cpu_reference_rate(aircraft, esteps, seed=1)
    t_total, kind, cores, alive = 0.0, "port", 1, 1.0
    for s in range(args.steps):
        rate, kind, cores, alive, dt, xf, st = cpu_reference_rate(aircraft, esteps, seed=0xF16 + s)
        t_total += dt
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, xf, st)
    value = aircraft * esteps * args.steps / t_total
    sample = f"{aircraft} aircraft x {esteps} Euler steps per bench step (of 2^20 x 10000), hifi xcg 0.25"
    line = {
        "impl": "reference", "metric": "hifi F-16 aircraft-steps/sec", "value": value, "unit": "aircraft-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "cfg2: 2^20-aircraft hifi batch, +-5% about trim, 10000 fused Euler steps (bounded sample)",
                   "aircraft_per_step": aircraft, "euler_steps_per_step": esteps, "dt": 0.001, "xcg": 0.25},
        "cpu_baseline": {"value": value, "unit": "aircraft-steps/s", "cores": cores, "kind": kind, "sample": sample,
                         "alive_fraction": alive},
        "e2e": {"value": value, "unit": "aircraft-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def measure_jacobians(L, ck, n, x_trim, u_trim, xcg, seed, scheme, reps=3):
    """Jacobians/s of linearise_batch_dev (A [18x18] + B [18x4] per trim point, env.py:294-342) on resident inputs:
    n perturbed-trim points, `reps` timed launches after one warm-up.  scheme 0 = forward (23 columns), 1 = central (44)."""
    x, u = perturbed_trim(n, x_trim, u_trim, seed, frac=0.02)
    d_x, d_u = L.f16_dev_alloc(x.nbytes), L.f16_dev_alloc(u.nbytes)
    d_A, d_B, d_st = L.f16_dev_alloc(n * 324 * 8), L.f16_dev_alloc(n * 72 * 8), L.f16_dev_alloc(4 * n)
    if not (d_x and d_u and d_A and d_B and d_st):
        raise RuntimeError("device allocation failed: " + L.f16_last_error().decode())
    ck(L.f16_memcpy_h2d(d_x, x.ctypes.data, x.nbytes), "h2d")
    ck(L.f16_memcpy_h2d(d_u, u.ctypes.data, u.nbytes), "h2d")

    def launch():
        ck(L.linearise_batch_dev(d_x, n, d_u, n, n, 1e-5, scheme, d_A, d_B, None, 1, None, xcg, d_st), "linearise_batch_dev")

    launch()
    ck(L.f16_sync(), "sync")
    ck(L.f16_timer_start(), "timer")
    for _ in range(reps):
        launch()
    ms = ctypes.c_float(0.0)
    ck(L.f16_timer_stop(ctypes.byref(ms)), "timer")
    st = np.zeros(n, dtype=np.int32)
    ck(L.f16_memcpy_d2h(st.ctypes.data, d_st, st.nbytes), "d2h")
    for p in (d_x, d_u, d_A, d_B, d_st):
        L.f16_dev_free(p)
    per_launch_ms = float(ms.value) / reps
    return {"value": n / (per_launch_ms * 1e-3), "unit": "Jacobian pairs (A 18x18, B 18x4)/s", "points": n,
            "scheme": "central" if scheme else "forward", "eps": 1e-5, "ms_per_launch": per_launch_ms,
            "valid_fraction": float((st == 0).mean()),
            "flop_per_jacobian": 32300.0 if scheme else 17200.0, "out_bytes_per_jacobian": 396 * 8}


def measure_cfg5(f16, L, ck, rank, n, ke, dt):
    """BASELINE cfg 5 at its stated size: n (default 8 Mi) aircraft per GPU -- 64 Mi on eight --, closed loop u = u0 - K (x - x_trim)
    fused into the step with the reference's own LQR gain (tests/golden K_lqr, env.py:344-358), hifi, xcg 0.35, +-5 % about
    trim, ke Euler steps in ONE launch on resident inputs.  One timed launch (seconds long) after a small warm-up launch of the
    same kernel; survivors counted on the device (f16_stats.cu)."""
    from f16_mpc_oop_py_b200.shard import rank_seed
    x_trim, u_trim, mpc_idx = trim_state("xcg35")
    K = -np.load(os.path.join(GOLDEN, "env_xcg35.npz"))["K_lqr"]
    law = f16.make_lqr(K, mpc_idx, x_trim[mpc_idx], u_trim, rows=[1, 2, 3])
    x, u = perturbed_trim(n, x_trim, u_trim, seed=rank_seed(0xC5, rank))
    d_x, d_u, d_st = L.f16_dev_alloc(x.nbytes), L.f16_dev_alloc(u.nbytes), L.f16_dev_alloc(4 * n)
    if not (d_x and d_u and d_st):
        raise RuntimeError("device allocation failed: " + L.f16_last_error().decode())
    ck(L.f16_memcpy_h2d(d_x, x.ctypes.data, x.nbytes), "h2d")
    ck(L.f16_memcpy_h2d(d_u, u.ctypes.data, u.nbytes), "h2d")
    nw = min(n, 1 << 18)   # warm-up: the same kernel on a corner of the batch, then the state is restored
    ck(L.step_batch_dev(d_x, n, d_u, n, nw, min(ke, 512), dt, ctypes.byref(law), None, 1, None, 0.35, d_st, None), "step_batch_dev")
    ck(L.f16_memcpy_h2d(d_x, x.ctypes.data, x.nbytes), "h2d")
    ck(L.f16_sync(), "sync")
    launches0 = L.f16_launch_count()
    ck(L.f16_timer_start(), "timer")
    ck(L.step_batch_dev(d_x, n, d_u, n, n, ke, dt, ctypes.byref(law), None, 1, None, 0.35, d_st, None), "step_batch_dev")
    ms = ctypes.c_float(0.0)
    ck(L.f16_timer_stop(ctypes.byref(ms)), "timer")
    launches = L.f16_launch_count() - launches0
    row = f16.state_summary_dev(d_x, n, n, d_st)
    for p in (d_x, d_u, d_st):
        L.f16_dev_free(p)
    return float(ms.value), row, int(launches)


# ---------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------
def run_ours(args):
    dist, rank, world, local = dist_setup(args.gpus)
    import f16_mpc_oop_py_b200 as f16
    L = f16.lib
    f16.init(device=local)
    L.f16_set_math_mode(f16.MATH_FAST if args.math == "fast" else f16.MATH_STRICT)
    if args.step_threads:
        L.f16_set_step_threads(args.step_threads)
    L.f16_set_table_staging(0 if args.no_table_staging else 1)

    n, ke = args.aircraft, args.euler_steps
    tag = "xcg35" if args.workload == "lqr" else "xcg25"
    xcg = 0.35 if args.workload == "lqr" else 0.25
    x_trim, u_trim, mpc_idx = trim_state(tag)
    from f16_mpc_oop_py_b200.shard import rank_seed
    x, u = perturbed_trim(n, x_trim, u_trim, seed=rank_seed(0xF16, rank))
    law = None
    if args.workload == "lqr":
        # BASELINE cfg 5: u = u0 - K (x - x_trim) on the reference's MPC states / inputs with the reference's own gain
        # (tests/golden: K_lqr = F16._calc_LQR_gain() = -dlqr(...), env.py:344-358, so the regulator gain is -K_lqr)
        K = -np.load(os.path.join(GOLDEN, f"env_{tag}.npz"))["K_lqr"]
        law = f16.make_lqr(K, mpc_idx, x_trim[mpc_idx], u_trim, rows=[1, 2, 3])
    law_p = ctypes.byref(law) if law is not None else None

    def ck(rc, what):
        if rc != 0:
            raise RuntimeError(f"{what}: {L.f16_last_error().decode()}")

    d_x0, d_x, d_u = L.f16_dev_alloc(x.nbytes), L.f16_dev_alloc(x.nbytes), L.f16_dev_alloc(u.nbytes)
    d_st = L.f16_dev_alloc(4 * n)
    if not (d_x0 and d_x and d_u and d_st):
        raise RuntimeError("device allocation failed: " + L.f16_last_error().decode())
    ck(L.f16_memcpy_h2d(d_x0, x.ctypes.data, x.nbytes), "h2d")
    ck(L.f16_memcpy_h2d(d_u, u.ctypes.data, u.nbytes), "h2d")

    # cudaMemcpy device-to-device on the library stream through its own symbol table (no CUDA binding needed)
    def reset_state():
        ck(L.f16_memcpy_d2d(d_x, d_x0, x.nbytes), "d2d")

    def one_step():
        reset_state()   # 144 MB device copy, > L2: every launch starts with cold inputs
        ck(L.step_batch_dev(d_x, n, d_u, n, n, ke, args.dt, law_p, None, 1, None, xcg, d_st, None), "step_batch_dev")

    # measured FP64 denominator (sustained DFMA rate of this GPU)
    peak = ctypes.c_double(0.0)
    ck(L.f16_measure_fp64_peak(300.0, ctypes.byref(peak)), "fp64 peak")

    for _ in range(args.warmup):
        one_step()
    ck(L.f16_sync(), "sync")

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if dist:
        dist.barrier()
    launches0 = L.f16_launch_count()
    ck(L.f16_timer_start(), "timer")
    for _ in range(args.steps):
        one_step()
    ms = ctypes.c_float(0.0)
    ck(L.f16_timer_stop(ctypes.byref(ms)), "timer")
    launches = L.f16_launch_count() - launches0
    if dist:
        dist.barrier()
    clocks = sampler.stop() if rank == 0 else None
    elapsed_ms = float(ms.value)

    st = np.zeros(n, dtype=np.int32)
    ck(L.f16_memcpy_d2h(st.ctypes.data, d_st, st.nbytes), "d2h")
    alive = float((st == 0).mean())
    xf = np.empty_like(x)
    ck(L.f16_memcpy_d2h(xf.ctypes.data, d_x, x.nbytes), "d2h")
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, xf, st, rank, world)

    # kernel-only duration of one launch (CUDA events on the launching stream), for the roofline
    reset_state()
    ck(L.f16_sync(), "sync")
    ck(L.f16_timer_start(), "timer")
    ck(L.step_batch_dev(d_x, n, d_u, n, n, ke, args.dt, law_p, None, 1, None, xcg, d_st, None), "step_batch_dev")
    kms = ctypes.c_float(0.0)
    ck(L.f16_timer_stop(ctypes.byref(kms)), "timer")
    kernel_ms = float(kms.value)

    # end-to-end through the host-buffer C ABI (what a ctypes user of the reference would call): H2D + kernels + D2H inside the
    # timed region, the call's own chunk pipeline overlapping them.  Twice: host arrays in pinned memory (f16_host_alloc_pinned)
    # and in ordinary pageable NumPy arrays (what a caller who knows nothing about CUDA hands over).
    hx = L.f16_host_alloc_pinned(x.nbytes)
    hu = L.f16_host_alloc_pinned(u.nbytes)
    hs = L.f16_host_alloc_pinned(4 * n)
    px = np.frombuffer((ctypes.c_double * (18 * n)).from_address(hx), dtype=np.float64).reshape(18, n)
    pu = np.frombuffer((ctypes.c_double * (4 * n)).from_address(hu), dtype=np.float64).reshape(4, n)
    gx, gu, gs = np.empty_like(x), np.empty_like(u), np.zeros(n, dtype=np.int32)

    def e2e_samples(bx, bu, ax, au, a_st):
        ms_l, wall_l = [], []
        for i in range(args.e2e_steps + 1):
            bx[:] = x
            bu[:] = u
            t0 = time.perf_counter()
            ck(L.f16_timer_start(), "timer")   # CUDA events on the library stream bracket the whole call
            ck(L.step_batch(ax, au, n, ke, args.dt, law_p, None, 1, None, xcg, a_st, None), "step_batch")
            ems = ctypes.c_float(0.0)
            ck(L.f16_timer_stop(ctypes.byref(ems)), "timer")
            if i > 0:   # the first call grows the library's device scratch
                ms_l.append(float(ems.value))
                wall_l.append(1e3 * (time.perf_counter() - t0))
        return ms_l, wall_l

    e2e_ms, e2e_wall = e2e_samples(px, pu, hx, hu, hs) if args.e2e_steps > 0 else ([], [])
    e2e_t = float(np.mean(e2e_ms)) if e2e_ms else float("nan")
    e2e_wall_t = float(np.mean(e2e_wall)) if e2e_wall else float("nan")
    e2e_equal = bool(np.array_equal(px, xf)) if e2e_ms else None
    pg_ms, pg_wall = e2e_samples(gx, gu, gx.ctypes.data, gu.ctypes.data, gs.ctypes.data) if args.e2e_steps > 0 else ([], [])
    pg_t = float(np.mean(pg_ms)) if pg_ms else float("nan")
    pg_equal = bool(np.array_equal(gx, xf)) if pg_ms else None
    for p in (hx, hu, hs):
        L.f16_host_free_pinned(p)

    jac = None
    if args.lin_variant is not None:
        L.f16_set_linearise_variant(args.lin_variant)
    jac_strict = None
    if not args.no_jacobians:
        jac = measure_jacobians(L, ck, args.jac_points, x_trim, u_trim, xcg, rank_seed(0x1AC, rank), 1)
        jac_fwd = measure_jacobians(L, ck, args.jac_points, x_trim, u_trim, xcg, rank_seed(0x1AC, rank), 0)
        for j in (jac, jac_fwd):
            j["kernel"] = ("linearise_fast_kernel (f16_fast.cuh arithmetic, two aircraft per warp)"
                           if args.math == "fast" and not args.lin_variant else "linearise_kernel (reference operation order, staged)")
        if args.math == "fast" and not args.lin_variant:   # the strict (parity-build) kernel beside it
            L.f16_set_linearise_variant(2)
            jac_strict = {"central": measure_jacobians(L, ck, args.jac_points, x_trim, u_trim, xcg, rank_seed(0x1AC, rank), 1),
                          "forward": measure_jacobians(L, ck, args.jac_points, x_trim, u_trim, xcg, rank_seed(0x1AC, rank), 0)}
            L.f16_set_linearise_variant(0)

    cfg5 = None
    if not args.no_cfg5 and args.workload == "open":
        if dist:
            dist.barrier()
        cfg5 = measure_cfg5(f16, L, ck, rank, args.cfg5_aircraft, ke, args.dt)

    # max over ranks (timings are the slowest rank's); the only collective: end-of-run statistics (SURVEY.md 8e)
    from f16_mpc_oop_py_b200 import shard
    dev = f"cuda:{local}" if dist else "cpu"
    if cfg5:
        c5_ms = shard.max_over_ranks(dist, [cfg5[0]], dev)[0]
        c5_sum = shard.gather_summaries(dist, cfg5[1], dev)
    elapsed_ms, kernel_ms, e2e_t, pg_t = shard.max_over_ranks(dist, [elapsed_ms, kernel_ms, e2e_t, pg_t], dev)
    # per-rank statistics reduced on the device (f16_stats.cu), then ONE all-gather of the 74-double rows
    summary = shard.gather_summaries(dist, f16.state_summary_dev(d_x, n, n, d_st), dev)
    alive = summary["alive_fraction"]

    total_steps = float(world) * n * ke * args.steps
    value = total_steps / (elapsed_ms * 1e-3)
    per_gpu_kernel = n * ke / (kernel_ms * 1e-3)
    flop = FLOP_PER_STEP["lqr" if law is not None else "open"]
    achieved_tf = per_gpu_kernel * flop / 1e12

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        rate, kind, cores, cpu_alive, _, _, _ = cpu_reference_rate(args.ref_aircraft, args.ref_euler_steps, seed=0xF16)
        cpu = {"value": rate, "unit": "aircraft-steps/s", "cores": cores, "kind": kind,
               "sample": f"{args.ref_aircraft} aircraft x {args.ref_euler_steps} Euler steps of the same workload",
               "alive_fraction": cpu_alive}

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        line = {
            "metric": "hifi F-16 aircraft-steps/sec", "value": value, "unit": "aircraft-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {
                "workload": ("cfg5: closed-loop LQR Monte Carlo, hifi xcg 0.35" if law is not None else
                             "cfg2: 2^20-aircraft hifi batch, +-5% about trim, 10000 fused Euler steps, xcg 0.25"),
                "aircraft_per_gpu": n, "euler_steps_per_step": ke, "dt": args.dt, "xcg": xcg, "math": args.math,
                "step_threads": args.step_threads or 384, "table_staging": "tma_smem" if not args.no_table_staging else "l2",
                "cold_inputs": "state re-copied from a 144 MB pristine buffer (> L2) before every launch",
                "alive_fraction": alive,
            },
            "roofline": {
                "bound": "fp64", "achieved": achieved_tf, "peak": float(peak.value), "unit": "TFLOP/s",
                "frac": achieved_tf / float(peak.value) if peak.value else None,
                "traffic": NCU_DRAM_BYTES_PER_LAUNCH.get((n, args.workload, args.math)), "traffic_unit": "bytes per launch (ncu dram read + write)",
                "kernel": "step_hifi_fast_kernel" if args.math == "fast" else "step_kernel", "kernel_ms": kernel_ms,
                "flop_per_aircraft_step": flop,
                "peak_source": "f16_measure_fp64_peak: DFMA micro-benchmark on this GPU in this run (MEASURED_PEAKS.json has no FP64 entry)",
                "hbm": {"achieved_gbs": n * BYTES_PER_AIRCRAFT_LAUNCH / (kernel_ms * 1e-3) / 1e9, "peak_gbs": hbm_peak,
                        "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback",
                        "bytes_per_aircraft_launch": BYTES_PER_AIRCRAFT_LAUNCH},
            },
            "e2e": {"value": float(world) * n * ke / (e2e_t * 1e-3), "unit": "aircraft-steps/s",
                    "h2d_bytes_per_step": int(x.nbytes + u.nbytes), "d2h_bytes_per_step": int(x.nbytes + 4 * n),
                    "ms_per_step": e2e_t, "host_wall_ms_per_step": e2e_wall_t, "bit_equal_to_device_path": e2e_equal,
                    "samples": len(e2e_ms), "samples_ms": e2e_ms, "host_memory": "pinned (f16_host_alloc_pinned)",
                    "pageable": {"value": float(world) * n * ke / (pg_t * 1e-3), "ms_per_step": pg_t, "samples": len(pg_ms),
                                 "samples_ms": pg_ms, "bit_equal_to_device_path": pg_equal,
                                 "host_memory": "ordinary NumPy arrays (pageable)"}},
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if jac:   # second half of BASELINE.json's metric; per-GPU figures of rank 0 (ranks run identical, independent work)
            peak_tf = float(peak.value)
            for j in (jac, jac_fwd):
                j["fp64_frac"] = j["value"] * j["flop_per_jacobian"] / 1e12 / peak_tf if peak_tf else None
                j["value_all_gpus"] = j["value"] * world
            line["jacobians"] = {"central": jac, "forward": jac_fwd}
            if jac_strict:
                for j in jac_strict.values():
                    j["fp64_frac"] = j["value"] * j["flop_per_jacobian"] / 1e12 / peak_tf if peak_tf else None
                    j["kernel"] = "linearise_kernel (reference operation order, staged): f16_set_linearise_variant(2)"
                line["jacobians"]["strict_build"] = jac_strict
        if cfg5:
            n5 = args.cfg5_aircraft
            per_gpu = n5 * ke / (c5_ms * 1e-3)
            line["cfg5_lqr"] = {
                "workload": "cfg5: closed-loop LQR Monte Carlo (u = u0 - K (x - x_trim) fused into the step, the reference's K_lqr), "
                            "hifi xcg 0.35, +-5% about trim",
                "aircraft_per_gpu": n5, "aircraft_total": n5 * world, "euler_steps": ke, "value": per_gpu * world,
                "unit": "aircraft-steps/s", "value_per_gpu": per_gpu, "ms_per_launch": c5_ms, "launches_per_gpu": cfg5[2],
                "alive_fraction": c5_sum["alive_fraction"], "flop_per_aircraft_step": FLOP_PER_STEP["lqr"],
                "fp64_frac": per_gpu * FLOP_PER_STEP["lqr"] / 1e12 / float(peak.value) if peak.value else None,
                "timing": "one launch on resident inputs, CUDA events, max over ranks",
            }
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    for p in (d_x0, d_x, d_u, d_st):
        L.f16_dev_free(p)
    if dist:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="open", choices=["open", "lqr"])
    ap.add_argument("--aircraft", type=int, default=1 << 20, help="aircraft per GPU")
    ap.add_argument("--euler-steps", type=int, default=10000, help="fused Euler steps per launch")
    ap.add_argument("--dt", type=float, default=0.001)
    ap.add_argument("--math", default="fast", choices=["strict", "fast"])
    ap.add_argument("--step-threads", type=int, default=0)
    ap.add_argument("--no-table-staging", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=3, help="timed step_batch() calls per kind of host memory")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-jacobians", action="store_true", help="skip the linearise_batch (Jacobians/s) measurement")
    ap.add_argument("--no-cfg5", action="store_true", help="skip the cfg-5 leg (closed-loop LQR Monte Carlo at 8 Mi aircraft per GPU)")
    ap.add_argument("--cfg5-aircraft", type=int, default=1 << 23, help="aircraft per GPU in the cfg-5 leg (8 Mi: 64 Mi on eight GPUs)")
    ap.add_argument("--jac-points", type=int, default=1 << 20,
                    help="trim points per GPU in the Jacobian measurement (SURVEY.md 8d: a 2^20-point batch for the throughput figure)")
    ap.add_argument("--lin-variant", type=int, default=None,
                    help="linearise kernel: 0 default (fast math: two aircraft per warp on the fast arithmetic), 1 strict warp per "
                         "aircraft, 2 strict CTA per 32 aircraft")
    ap.add_argument("--ref-aircraft", type=int, default=4096, help="aircraft in the CPU sample")
    ap.add_argument("--ref-euler-steps", type=int, default=200, help="Euler steps in the CPU sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's final state and status words as DIR/x.npy and DIR/status.npy "
                         f"(x.rank<k>.npy, status.rank<k>.npy per rank; a fixed sample of {DUMP_AIRCRAFT} aircraft over all ranks "
                         "of a larger batch); bench_outputs/ in the repository is ignored by git")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return run_reference(args) if args.impl == "reference" else run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
