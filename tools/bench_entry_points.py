#!/usr/bin/env python3
"""Time every device entry point of libf16_b200.so over a range of batch sizes (CUDA events on the library stream,
inputs resident in HBM, an L2 flush before every timed launch) and print one JSON line per (entry point, N) with the
roofline that bounds it:

  Nlplant_batch_dev / calc_xdot_batch_dev   HBM: (17+18) / (18+4+18) doubles per aircraft
  step_batch_dev K=1                        HBM: 320 B per aircraft
  linearise_batch_dev                       FP64 (17.2 k / 32.3 k flop per Jacobian pair) and HBM (3168 B written)
  trim_batch_dev                            objective evaluations/s
  state_summary_batch_dev                   HBM: 152 B per aircraft (one pass: 18 planes + the status words per group of six states)

Usage: python tools/bench_entry_points.py [--math strict|fast] [--sizes 4096,65536,1048576] [--reps 5] [--staging 0|1]
"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from bench import perturbed_trim, trim_state  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--math", default="fast", choices=["strict", "fast"])
    ap.add_argument("--sizes", default="4736,56832,1048576")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--staging", type=int, default=1)
    ap.add_argument("--fi", type=int, default=1)
    ap.add_argument("--only", default="")
    ap.add_argument("--no-flush", action="store_true")
    args = ap.parse_args()
    import f16_mpc_oop_py_b200 as f16
    L = f16.lib
    f16.init(device=0)
    L.f16_set_math_mode(f16.MATH_FAST if args.math == "fast" else f16.MATH_STRICT)
    L.f16_set_table_staging(args.staging)
    try:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
    except OSError:
        peaks = {}
    hbm = peaks.get("hbm_gbs", 6650.0)
    pk = ctypes.c_double(0.0)
    L.f16_measure_fp64_peak(200.0, ctypes.byref(pk))
    fp64 = pk.value

    def ck(rc, what):
        if rc != 0:
            raise RuntimeError(f"{what}: {L.f16_last_error().decode()}")

    def timed(fn):
        fn()
        ck(L.f16_sync(), "sync")
        best, tot = None, 0.0
        for _ in range(args.reps):
            if not args.no_flush:
                ck(L.f16_flush_l2(), "flush")
            ck(L.f16_timer_start(), "timer")
            fn()
            ms = ctypes.c_float(0.0)
            ck(L.f16_timer_stop(ctypes.byref(ms)), "timer")
            tot += ms.value
            best = ms.value if best is None else min(best, ms.value)
        return best, tot / args.reps

    tag = "xcg25" if args.fi else "lofi_xcg25"
    x_trim, u_trim, _ = trim_state(tag)
    only = set(args.only.split(",")) if args.only else None
    for n in [int(s) for s in args.sizes.split(",")]:
        x, u = perturbed_trim(n, x_trim, u_trim, seed=7, frac=0.02)
        d_x, d_u, d_o = L.f16_dev_alloc(x.nbytes), L.f16_dev_alloc(u.nbytes), L.f16_dev_alloc(x.nbytes)
        d_st = L.f16_dev_alloc(4 * n)
        ck(L.f16_memcpy_h2d(d_x, x.ctypes.data, x.nbytes), "h2d")
        ck(L.f16_memcpy_h2d(d_u, u.ctypes.data, u.nbytes), "h2d")
        common = {"N": n, "math": args.math, "staging": args.staging, "fi": args.fi}

        def report(name, best, avg, nbytes=None, flop=None, units=None, unit_name=None):
            r = dict(common, entry=name, ms_best=round(best, 5), ms_avg=round(avg, 5))
            if nbytes:
                r["GBs"] = round(nbytes / (best * 1e-3) / 1e9, 1)
                r["hbm_frac"] = round(r["GBs"] / hbm, 4)
            if flop:
                r["TFLOPs"] = round(flop / (best * 1e-3) / 1e12, 3)
                r["fp64_frac"] = round(r["TFLOPs"] / fp64, 4)
            if units:
                r[unit_name] = units / (best * 1e-3)
            print(json.dumps(r), flush=True)

        if not only or "nlplant" in only:
            b, a = timed(lambda: ck(L.Nlplant_batch_dev(d_x, n, d_o, n, None, args.fi, None, 0.25, n, d_st), "nlplant"))
            report("Nlplant_batch_dev", b, a, nbytes=n * (35 * 8 + 4), flop=n * 710.0, units=n, unit_name="evals_per_s")
        if not only or "calc_xdot" in only:
            b, a = timed(lambda: ck(L.calc_xdot_batch_dev(d_x, n, d_u, n, d_o, n, None, args.fi, None, 0.25, n, d_st), "xdot"))
            report("calc_xdot_batch_dev", b, a, nbytes=n * (40 * 8 + 4), flop=n * 715.0, units=n, unit_name="evals_per_s")
        if not only or "step1" in only:
            ck(L.f16_memcpy_d2d(d_o, d_x, x.nbytes), "d2d")
            b, a = timed(lambda: ck(L.step_batch_dev(d_o, n, d_u, n, n, 1, 0.0, None, None, args.fi, None, 0.25, d_st, None), "step"))
            report("step_batch_dev K=1", b, a, nbytes=n * (40 * 8 + 4), flop=n * 750.0, units=n, unit_name="steps_per_s")
        if not only or "step100" in only:
            ck(L.f16_memcpy_d2d(d_o, d_x, x.nbytes), "d2d")
            b, a = timed(lambda: ck(L.step_batch_dev(d_o, n, d_u, n, n, 100, 0.0, None, None, args.fi, None, 0.25, d_st, None), "step"))
            report("step_batch_dev K=100", b, a, nbytes=n * (40 * 8 + 4), flop=n * 75000.0, units=n * 100, unit_name="steps_per_s")
        if not only or "summary" in only:
            row = np.empty(74)
            b, a = timed(lambda: ck(L.state_summary_batch_dev(d_x, n, n, None, row.ctypes.data), "summary"))
            report("state_summary_batch_dev (one pass + 592 B D2H)", b, a, nbytes=n * 152, units=n, unit_name="aircraft_per_s")
            # with status words: every aircraft alive (the first-survivor search stops at once), and only the last one alive
            # (the search reads every status word)
            for name, last_only in (("all alive", False), ("one survivor, the last", True)):
                st = np.zeros(n, dtype=np.int32)
                if last_only:
                    st[:-1] = 4
                ck(L.f16_memcpy_h2d(d_st, st.ctypes.data, st.nbytes), "h2d")
                b, a = timed(lambda: ck(L.state_summary_batch_dev(d_x, n, n, d_st, row.ctypes.data), "summary"))
                report(f"state_summary_batch_dev, status: {name}", b, a, nbytes=n * 152, units=n, unit_name="aircraft_per_s")
        if (not only or "linearise" in only) and n <= (1 << 18):
            d_A, d_B = L.f16_dev_alloc(n * 324 * 8), L.f16_dev_alloc(n * 72 * 8)
            for scheme, nm, fl in ((0, "forward", 17200.0), (1, "central", 32300.0)):
                b, a = timed(lambda: ck(L.linearise_batch_dev(d_x, n, d_u, n, n, 1e-5, scheme, d_A, d_B, None, args.fi, None, 0.25, d_st), "lin"))
                report(f"linearise_batch_dev {nm}", b, a, nbytes=n * (396 + 22) * 8, flop=n * fl, units=n, unit_name="jacobians_per_s")
            L.f16_dev_free(d_A)
            L.f16_dev_free(d_B)
        if (not only or "trim" in only) and n <= (1 << 17):
            r = np.random.default_rng(3)
            h = r.uniform(5000, 40000, n)
            v = r.uniform(300, 900, n)
            d_h, d_v, d_info = L.f16_dev_alloc(8 * n), L.f16_dev_alloc(8 * n), L.f16_dev_alloc(32 * n)
            ck(L.f16_memcpy_h2d(d_h, h.ctypes.data, 8 * n), "h2d")
            ck(L.f16_memcpy_h2d(d_v, v.ctypes.data, 8 * n), "h2d")
            b, a = timed(lambda: ck(L.trim_batch_dev(d_h, d_v, n, 1e-10, 50000, None, d_o, n, d_info, n, None, args.fi, None, 0.25, d_st), "trim"))
            info = np.zeros((4, n))
            ck(L.f16_memcpy_d2h(info.ctypes.data, d_info, info.nbytes), "d2h")
            report("trim_batch_dev", b, a, units=float(info[2].sum()), unit_name="objective_evals_per_s")
            for p in (d_h, d_v, d_info):
                L.f16_dev_free(p)
        for p in (d_x, d_u, d_o, d_st):
            L.f16_dev_free(p)


if __name__ == "__main__":
    main()
