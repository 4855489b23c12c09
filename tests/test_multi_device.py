"""The host-buffer entry points as pipelines of chunks and as slices over several device contexts (include/f16_b200.h:
f16_init_devices, f16_set_host_pipeline).  Aircraft never interact (SURVEY.md 8e), so neither the cut into chunks nor the
cut into per-device slices may change a single bit of any per-aircraft result; the statistics rows are merged on the host by
Chan's update and agree to rounding.  On a one-GPU box the slices run on two contexts of the same GPU (an ordinal may be listed
twice), which exercises the same slicing, threading and merging code as two GPUs do."""
import ctypes

import numpy as np
import pytest

from _inputs import perturbed_trim
from conftest import load_golden

pytestmark = pytest.mark.gpu


def _batch(n, seed=5):
    g = load_golden("xcg25")
    x, u = perturbed_trim(n, g["x_trim"], seed=seed, frac=0.05)
    r = np.random.default_rng(seed)
    fi = (r.uniform(size=n) < 0.7).astype(np.uint8)           # mixed hifi / lofi
    xcg = np.where(r.uniform(size=n) < 0.5, 0.25, 0.35)
    return x, u, fi, xcg


def _run_all(f16, n_step, n_lin, n_trim):
    """every sliced entry point once; returns a dict of outputs"""
    out = {}
    x, u, fi, xcg = _batch(n_step)
    fb = f16.F16Batch(x, u, fi_flag=fi, xcg=xcg)
    out["xdot"] = fb._calc_xdot(x, u)
    out["xdot_st"] = fb.last_status.copy()
    fb.step(K=3)
    out["x3"], out["st3"], out["k3"] = fb.x.copy(), fb.status.copy(), fb.steps_done.copy()
    fb.step(K=20)                                               # mixed batch, K >= 8: the fidelity partition on every chunk
    out["x23"], out["st23"] = fb.x.copy(), fb.status.copy()
    fb = f16.F16Batch(x, u, xcg=0.25)                           # uniform hifi, long run: the time-chunked step kernel
    fb.step(K=600)
    out["x600"], out["st600"] = fb.x.copy(), fb.status.copy()
    out["nl"], out["nl_st"] = f16.nlplant(np.ascontiguousarray(x[:17]), fi=fi, xcg=xcg)
    fb = f16.F16Batch(x[:, :n_lin], u[:, :n_lin], fi_flag=fi[:n_lin], xcg=xcg[:n_lin])
    out["A"], out["B"], _, _ = fb.linearise(fb.x, fb.u, scheme="central")
    out["lin_st"] = fb.last_status.copy()
    fb = f16.F16Batch(x[:, :n_lin], u[:, :n_lin], xcg=0.35)
    out["traj"] = fb.rollout(K=40, snap_every=10).copy()
    out["traj_x"] = fb.x.copy()
    fb = f16.F16Batch(x, u, xcg=0.35)
    out["rows"] = fb.rollout_stats(K=40, snap_every=20).copy()
    out["rows_x"] = fb.x.copy()
    out["summary"] = f16.state_summary(fb.x, fb.status)
    r = np.random.default_rng(3)
    h, v = r.uniform(5000, 30000, n_trim), r.uniform(400, 800, n_trim)
    xt, opt = f16.trim(h, v, tol=1e-10, maxiter=3000, xcg=0.35)
    out["trim"], out["trim_fun"], out["trim_nit"], out["trim_st"] = xt, opt["fun"], opt["nit"], opt["status"]
    return out


EXACT = ["xdot", "xdot_st", "x3", "st3", "k3", "x23", "st23", "x600", "st600", "nl", "nl_st", "A", "B", "lin_st", "traj", "traj_x",
         "rows_x", "trim", "trim_fun", "trim_nit", "trim_st"]


def _compare(a, b):
    for k in EXACT:
        assert np.array_equal(a[k], b[k], equal_nan=True), k
    for k in ("rows", "summary"):   # counts, min and max exactly; mean / M2 to rounding (another summation order)
        ra, rb = np.asarray(a[k]).reshape(-1, 74), np.asarray(b[k]).reshape(-1, 74)
        assert np.array_equal(ra[:, :38], rb[:, :38]), k
        assert np.allclose(ra[:, 38:56], rb[:, 38:56], rtol=1e-12, atol=1e-300), k
        assert np.allclose(ra[:, 56:], rb[:, 56:], rtol=1e-9, atol=1e-18), k


@pytest.mark.parametrize("math", ["fast", "strict"])
def test_chunk_pipeline_does_not_change_a_bit(f16, math):
    """300 001 aircraft (ragged: not a multiple of 32 or of the chunk size) = 4 chunks of the one-shot calls and of the K = 3
    step, 1 of the K = 600 step; against the same calls as ONE chunk (f16_set_host_pipeline(0))."""
    prev_math = f16.lib.f16_set_math_mode(f16.MATH_FAST if math == "fast" else f16.MATH_STRICT)
    try:
        prev = f16.lib.f16_set_host_pipeline(0)
        one = _run_all(f16, 300_001, 40_003, 300)
        f16.lib.f16_set_host_pipeline(1)
        piped = _run_all(f16, 300_001, 40_003, 300)
        f16.lib.f16_set_host_pipeline(prev)
        _compare(one, piped)
    finally:
        f16.lib.f16_set_math_mode(prev_math)


def test_slices_over_device_contexts_equal_one_context(f16):
    """f16_init_devices: the same calls on one context and on 2 (and 3) contexts -- real GPUs where the box has them, else
    contexts of the same GPU -- give the same bits."""
    import torch
    ngpu = torch.cuda.device_count()
    prev_math = f16.lib.f16_set_math_mode(f16.MATH_FAST)
    try:
        assert f16.lib.f16_device_count() == 1
        one = _run_all(f16, 200_003, 30_001, 5000)
        for devs in ([0, 1 % ngpu], [0, 1 % ngpu, 2 % ngpu]):
            f16.shutdown()
            assert f16.lib.f16_device_count() == 0
            assert f16.init_devices(devs) == len(devs)
            # a second init on another list is refused, the same list is accepted
            arr = (ctypes.c_int * 1)(0)
            assert f16.lib.f16_init_devices(None, arr, 1) == -3
            assert f16.init_devices(devs) == len(devs)
            many = _run_all(f16, 200_003, 30_001, 5000)
            _compare(one, many)
            # the *_dev entry points follow f16_use_device
            for i in range(len(devs)):
                assert f16.lib.f16_use_device(i) >= 0
                assert f16.lib.f16_device() == devs[i]
                x, u, _, _ = _batch(4096, seed=9)
                fb = f16.F16Batch(x, u, xcg=0.25)
                s = f16.state_summary(fb.x, fb.status)
                assert s[0] == 4096
            assert f16.lib.f16_use_device(len(devs)) == -3
            f16.lib.f16_use_device(0)
    finally:
        f16.shutdown()
        f16.init()
        f16.lib.f16_set_math_mode(prev_math)


@pytest.mark.parametrize("math", ["fast", "strict"])
def test_survivor_compaction_equals_one_launch(f16, math):
    """A Monte-Carlo run with casualties: xcg 0.35 open loop, +-5 % about trim, 5 s -- a third of the batch leaves the envelope.
    With f16_set_step_compaction(1) the run is eight chunks of steps with the survivors repacked in between; states, status
    words and step counts must be the bits of the single launch, with and without per-aircraft xcg / steps_done arrays, through
    the host entry point (chunk pipeline) and the device entry point."""
    g = load_golden("xcg35")
    n, K = 140_001, 5000 if math == "fast" else 4096
    x, u = perturbed_trim(n, g["x_trim"], seed=11, frac=0.05)
    xcg = np.full(n, 0.35)
    prev_math = f16.lib.f16_set_math_mode(f16.MATH_FAST if math == "fast" else f16.MATH_STRICT)
    prev = f16.lib.f16_set_step_compaction(0)
    try:
        ref = f16.F16Batch(x, u, xcg=0.35)
        ref.step(K=K)
        dead = (ref.status != 0).mean()
        assert 0.1 < dead < 0.9, dead          # the run does lose aircraft, and keeps some
        f16.lib.f16_set_step_compaction(1)
        for xc in (0.35, xcg):
            fb = f16.F16Batch(x, u, xcg=xc)
            fb.step(K=K)
            assert np.array_equal(fb.x, ref.x, equal_nan=True)
            assert np.array_equal(fb.status, ref.status) and np.array_equal(fb.steps_done, ref.steps_done)
        # device entry point, no steps_done array
        L = f16.lib
        d_x, d_u, d_st = L.f16_dev_alloc(x.nbytes), L.f16_dev_alloc(u.nbytes), L.f16_dev_alloc(4 * n)
        assert L.f16_memcpy_h2d(d_x, x.ctypes.data, x.nbytes) == 0 and L.f16_memcpy_h2d(d_u, u.ctypes.data, u.nbytes) == 0
        assert L.step_batch_dev(d_x, n, d_u, n, n, K, 0.001, None, None, 1, None, 0.35, d_st, None) == 0
        xo, so = np.empty_like(x), np.zeros(n, np.int32)
        assert L.f16_memcpy_d2h(xo.ctypes.data, d_x, x.nbytes) == 0 and L.f16_memcpy_d2h(so.ctypes.data, d_st, 4 * n) == 0
        for p in (d_x, d_u, d_st):
            L.f16_dev_free(p)
        assert np.array_equal(xo, ref.x, equal_nan=True) and np.array_equal(so, ref.status)
    finally:
        f16.lib.f16_set_step_compaction(prev)
        f16.lib.f16_set_math_mode(prev_math)


@pytest.mark.parametrize("math", ["fast", "strict"])
def test_device_entry_points_stay_inside_their_arrays(f16, math):
    """compute-sanitizer is not available on the GPU pool: canaries instead.  Every *_dev entry point runs on arrays whose
    planes are wider than the batch (plane stride ld > N, odd -- no tensor map, plain loads -- and even -- TMA boxes), in a
    buffer with a guard band behind the last plane; the padding columns, the guard bands and the inputs must come back
    bit for bit, for ragged batch sizes around the warp / CTA / chunk boundaries."""
    L = f16.lib
    prev_math = L.f16_set_math_mode(f16.MATH_FAST if math == "fast" else f16.MATH_STRICT)
    prev_comp = L.f16_set_step_compaction(1)
    CANARY = -1.2345678901234567e+300
    g = load_golden("xcg35")

    def dev(a):
        p = L.f16_dev_alloc(a.nbytes)
        assert p and L.f16_memcpy_h2d(p, a.ctypes.data, a.nbytes) == 0
        return p

    def back(p, like):
        out = np.empty_like(like)
        assert L.f16_memcpy_d2h(out.ctypes.data, p, like.nbytes) == 0
        return out

    try:
        for n, pad, K in ((1, 3, 1), (31, 1, 2), (4097, 37, 1), (4097, 64, 7), (70_001, 64, 1), (70_001, 37, 9), (66_000, 64, 4096)):
            ld = n + pad
            x, u = perturbed_trim(n, g["x_trim"], seed=n, frac=0.05)
            X = np.full((19, ld), CANARY); X[:18, :n] = x          # plane 18 = guard band
            U = np.full((5, ld), CANARY); U[:4, :n] = u
            O = np.full((19, ld), CANARY)
            ST = np.full(ld + 64, 0x5A5A5A5A, dtype=np.int32)
            KD = np.full(ld + 64, 0x5A5A5A5A, dtype=np.int32)
            d_x, d_u, d_o, d_st, d_k = dev(X), dev(U), dev(O), dev(ST), dev(KD)
            # calc_xdot / Nlplant: outputs in O, inputs untouched
            assert L.calc_xdot_batch_dev(d_x, ld, d_u, ld, d_o, ld, None, 1, None, 0.35, n, d_st) == 0
            o = back(d_o, O)
            assert np.all(o[:18, n:] == CANARY) and np.all(o[18] == CANARY) and np.isfinite(o[:18, :n]).all()
            assert L.Nlplant_batch_dev(d_x, ld, d_o, ld, None, 1, None, 0.35, n, d_st) == 0
            o = back(d_o, O)
            assert np.all(o[:18, n:] == CANARY) and np.all(o[18] == CANARY)
            assert np.array_equal(back(d_x, X), X) and np.array_equal(back(d_u, U), U)
            # linearise (small n only: 3 KB of output per aircraft)
            if n <= 4097:
                A = np.full((n + 2, 324), CANARY); B = np.full((n + 2, 72), CANARY)
                d_a, d_b = dev(A), dev(B)
                assert L.linearise_batch_dev(d_x, ld, d_u, ld, n, 1e-5, 1, d_a, d_b, None, 1, None, 0.35, d_st) == 0
                a, b = back(d_a, A), back(d_b, B)
                assert np.all(a[n:] == CANARY) and np.all(b[n:] == CANARY) and np.isfinite(a[:n]).all() and np.isfinite(b[:n]).all()
                L.f16_dev_free(d_a); L.f16_dev_free(d_b)
            # the step: state advanced in place, nothing else touched
            assert L.step_batch_dev(d_x, ld, d_u, ld, n, K, 0.001, None, None, 1, None, 0.35, d_st, d_k) == 0
            x1, st, kd = back(d_x, X), back(d_st, ST), back(d_k, KD)
            assert np.all(x1[:18, n:] == CANARY) and np.all(x1[18] == CANARY) and np.array_equal(back(d_u, U), U)
            assert np.all(st[n:] == 0x5A5A5A5A) and np.all(kd[n:] == 0x5A5A5A5A)
            assert np.all((kd[:n] == K) | (st[:n] != 0)) and np.isfinite(x1[:18, :n]).all()
            row = f16.state_summary_dev(d_x, ld, n, d_st)
            assert row[0] == n and row[1] == (st[:n] == 0).sum()
            for p in (d_x, d_u, d_o, d_st, d_k):
                L.f16_dev_free(p)
    finally:
        L.f16_set_step_compaction(prev_comp)
        L.f16_set_math_mode(prev_math)


def test_host_entry_points_stay_inside_their_arrays(f16):
    """the same for the host-buffer calls (chunk pipeline, 2-D copies into slices of the caller's planes): guard bands behind
    every output array, a ragged batch of 300 001 aircraft = four chunks"""
    L = f16.lib
    prev_math = L.f16_set_math_mode(f16.MATH_FAST)
    CANARY, GUARD = -1.2345678901234567e+300, 4096
    try:
        g = load_golden("xcg25")
        n = 300_001
        x, u = perturbed_trim(n, g["x_trim"], seed=4, frac=0.05)

        def guarded(a):
            buf = np.full(a.size + GUARD, CANARY)
            buf[:a.size] = a.ravel()
            return buf

        def vp(a):
            return ctypes.c_void_p(a.ctypes.data)

        X, U, O = guarded(x), guarded(u), np.full(18 * n + GUARD, CANARY)
        ST = np.full(n + GUARD, 0x5A5A5A5A, dtype=np.int32)
        KD = np.full(n + GUARD, 0x5A5A5A5A, dtype=np.int32)
        assert L.calc_xdot_batch(vp(X), vp(U), vp(O), None, 1, None, 0.25, n, vp(ST)) == 0
        assert np.all(O[18 * n:] == CANARY) and np.isfinite(O[:18 * n]).all() and np.all(ST[n:] == 0x5A5A5A5A)
        assert np.array_equal(X[:18 * n], x.ravel()) and np.all(X[18 * n:] == CANARY) and np.all(U[4 * n:] == CANARY)
        O[:] = CANARY
        assert L.Nlplant_batch(vp(X), vp(O), None, 1, None, 0.25, n, vp(ST)) == 0
        assert np.all(O[18 * n:] == CANARY) and np.all(ST[n:] == 0x5A5A5A5A)
        for K in (1, 600):
            X = guarded(x)
            assert L.step_batch(vp(X), vp(U), n, K, 0.001, None, None, 1, None, 0.25, vp(ST), vp(KD)) == 0
            assert np.all(X[18 * n:] == CANARY) and np.all(U[4 * n:] == CANARY) and np.array_equal(U[:4 * n], u.ravel())
            assert np.all(ST[n:] == 0x5A5A5A5A) and np.all(KD[n:] == 0x5A5A5A5A) and np.all(KD[:n] == K)
        m = 40_003
        A, B = np.full(m * 324 + GUARD, CANARY), np.full(m * 72 + GUARD, CANARY)
        xs, us = np.ascontiguousarray(x[:, :m]), np.ascontiguousarray(u[:, :m])
        assert L.linearise_batch(vp(xs), vp(us), m, 1e-5, 0, vp(A), vp(B), None, 1, None, 0.25, vp(ST)) == 0
        assert np.all(A[m * 324:] == CANARY) and np.all(B[m * 72:] == CANARY) and np.isfinite(A[:m * 324]).all()
        t = 5000
        h, v = np.linspace(5000, 30000, t), np.linspace(400, 800, t)
        XT, INFO = np.full(18 * t + GUARD, CANARY), np.full(4 * t + GUARD, CANARY)
        assert L.trim_batch(vp(h), vp(v), t, 1e-10, 3000, None, vp(XT), vp(INFO), None, 1, None, 0.35, vp(ST)) == 0
        assert np.all(XT[18 * t:] == CANARY) and np.all(INFO[4 * t:] == CANARY) and np.isfinite(XT[:18 * t]).all()
    finally:
        L.f16_set_math_mode(prev_math)


def test_entry_points_from_concurrent_host_threads(f16):
    """two host threads hammer different entry points at once (ctypes releases the GIL; the library serialises on its mutex):
    every call returns the result of the same call made alone"""
    import threading
    g = load_golden("xcg25")
    x, u = perturbed_trim(50_001, g["x_trim"], seed=8, frac=0.05)
    prev = f16.lib.f16_set_math_mode(f16.MATH_FAST)
    try:
        fb = f16.F16Batch(x, u, xcg=0.25)
        ref_xd = fb._calc_xdot(x, u)
        fb.step(K=50)
        ref_x = fb.x.copy()
        bad = []

        def derivs():
            b = f16.F16Batch(x, u, xcg=0.25)
            for _ in range(15):
                if not np.array_equal(b._calc_xdot(x, u), ref_xd):
                    bad.append("calc_xdot")

        def steps():
            for _ in range(15):
                b = f16.F16Batch(x, u, xcg=0.25)
                b.step(K=50)
                if not np.array_equal(b.x, ref_x):
                    bad.append("step")

        ts = [threading.Thread(target=derivs), threading.Thread(target=steps), threading.Thread(target=derivs)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        assert not bad, bad
    finally:
        f16.lib.f16_set_math_mode(prev)


# ---- argument checks --------------------------------------------------------------------------------------------------
# Every host-buffer and *_dev entry point (the linalg calls: tests/test_linalg.py) as (arguments, pointers that must not be
# NULL when N > 0, further rejected values, what N = 0 does).  Array arguments are ("f8" | "i4" | "u1", count) and are filled with
# canaries; a _dev entry point gets device copies of them, except for the ("host", ...) ones, which the ABI takes on the host.
def _sel(n):
    return [("fi", ("u1", n)), ("fi_default", 1), ("xcg", ("f8", n)), ("xcg_default", 0.25)]


_BAD_LAWS = [{"lqr": ("law", 19, 0)}, {"lqr": ("law", -1, 0)}, {"lqr": ("law", 1, 18)}, {"lqr": ("law", 1, -1)}]
_STEP_BAD = [{"K": -1}] + _BAD_LAWS
_SNAP_BAD = _STEP_BAD + [{"snap_every": 0}]
_LIN_BAD = [{"scheme": 2}, {"scheme": -1}, {"eps": 1e-13}, {"eps": 2e3}, {"eps": float("nan")}]
_TRIM_BAD = [{"tol": -1.0}, {"tol": float("nan")}, {"maxiter": 0}]
_ENTRY = {
    "Nlplant_batch": (lambda n: [("xu", ("f8", 17 * n)), ("xdot", ("f8", 18 * n))] + _sel(n) + [("N", n), ("status", ("i4", n))],
                      ["xu", "xdot"], [], "ok"),
    "calc_xdot_batch": (lambda n: [("x", ("f8", 18 * n)), ("u", ("f8", 4 * n)), ("xdot", ("f8", 18 * n))] + _sel(n) +
                        [("N", n), ("status", ("i4", n))], ["x", "u", "xdot"], [], "ok"),
    "step_batch": (lambda n: [("x", ("f8", 18 * n)), ("u", ("f8", 4 * n)), ("N", n), ("K", 2), ("dt", 1e-3), ("lqr", None)] + _sel(n) +
                   [("status", ("i4", n)), ("steps", ("i4", n))], ["x", "u"], _STEP_BAD, "ok"),
    "step_batch_traj": (lambda n: [("x", ("f8", 18 * n)), ("u", ("f8", 4 * n)), ("N", n), ("K", 4), ("snap_every", 2), ("dt", 1e-3),
                                   ("lqr", None)] + _sel(n) + [("traj", ("f8", 2 * 18 * n)), ("status", ("i4", n))],
                        ["x", "u", "traj"], _SNAP_BAD, "ok"),
    "linearise_batch": (lambda n: [("x", ("f8", 18 * n)), ("u", ("f8", 4 * n)), ("N", n), ("eps", 1e-5), ("scheme", 0),
                                   ("A", ("f8", 324 * n)), ("B", ("f8", 72 * n))] + _sel(n) + [("status", ("i4", n))],
                        ["x", "u", "A", "B"], _LIN_BAD, "ok"),
    "trim_batch": (lambda n: [("h", ("f8", n)), ("V", ("f8", n)), ("N", n), ("tol", 1e-10), ("maxiter", 100), ("ux0", None),
                              ("x_trim", ("f8", 18 * n)), ("info", ("f8", 4 * n))] + _sel(n) + [("status", ("i4", n))],
                   ["h", "V", "x_trim"], _TRIM_BAD, "ok"),
    "step_batch_stats": (lambda n: [("x", ("f8", 18 * n)), ("u", ("f8", 4 * n)), ("N", n), ("K", 4), ("snap_every", 2), ("dt", 1e-3),
                                    ("lqr", None)] + _sel(n) + [("rows", ("f8", 2 * 74)), ("status", ("i4", n))],
                         ["x", "u", "rows"], _SNAP_BAD, "rows"),
    "state_summary_batch": (lambda n: [("x", ("f8", 18 * n)), ("N", n), ("status", ("i4", n)), ("row", ("f8", 74))],
                            ["x", "row"], [], "rows"),
    "lqr_gain_batch": (lambda n: [("x", ("f8", 18 * n)), ("u", ("f8", 4 * n)), ("N", n), ("dt", 0.02), ("K", ("f8", 27 * n))] +
                       _sel(n) + [("status", ("i4", n))], ["x", "u", "K"], [{"dt": 0.0}, {"dt": float("nan")}], "ok"),
    "f16_hifi_probe": (lambda n: [("a", ("f8", n)), ("b", ("f8", n)), ("el", ("f8", n)), ("N", n), ("coef", ("f8", 44 * n)),
                                  ("cells", ("i4", 8 * n)), ("status", ("i4", n))], ["a", "b", "el", "coef", "cells"], [], "arg"),
    "f16_fast_probe": (lambda n: [("a", ("f8", n)), ("b", ("f8", n)), ("el", ("f8", n)), ("N", n), ("coef", ("f8", 44 * n)),
                                  ("cells", ("i4", 4 * n)), ("lam", ("f8", 4 * n)), ("status", ("i4", n))],
                       ["a", "b", "el", "coef", "cells", "lam"], [], "arg"),
    "f16_lofi_probe": (lambda n: [("a", ("f8", n)), ("b", ("f8", n)), ("el", ("f8", n)), ("dail", ("f8", n)), ("drud", ("f8", n)),
                                  ("N", n), ("out", ("f8", 19 * n))], ["a", "b", "el", "dail", "drud", "out"], [], "arg"),
    "f16_div_probe": (lambda n: [("a", ("f8", n)), ("b", ("f8", n)), ("N", n), ("out", ("f8", 3 * n))], ["a", "b", "out"], [], "arg"),
    "atmos_batch": (lambda n: [("alt", ("f8", n)), ("vt", ("f8", n)), ("N", n), ("coeff", ("f8", 3 * n))], ["alt", "vt", "coeff"],
                    [], "arg"),
    "Nlplant_batch_dev": (lambda n: [("xu", ("f8", 17 * n)), ("ld_in", n), ("xdot", ("f8", 18 * n)), ("ld_out", n)] + _sel(n) +
                          [("N", n), ("status", ("i4", n))], ["xu", "xdot"], [{"ld_in": 63}, {"ld_out": 63}], "ok"),
    "calc_xdot_batch_dev": (lambda n: [("x", ("f8", 18 * n)), ("ld_x", n), ("u", ("f8", 4 * n)), ("ld_u", n), ("xdot", ("f8", 18 * n)),
                                       ("ld_out", n)] + _sel(n) + [("N", n), ("status", ("i4", n))],
                            ["x", "u", "xdot"], [{"ld_x": 63}, {"ld_u": 63}, {"ld_out": 63}], "ok"),
    "step_batch_dev": (lambda n: [("x", ("f8", 18 * n)), ("ld_x", n), ("u", ("f8", 4 * n)), ("ld_u", n), ("N", n), ("K", 2),
                                  ("dt", 1e-3), ("lqr", None)] + _sel(n) + [("status", ("i4", n)), ("steps", ("i4", n))],
                       ["x", "u"], _STEP_BAD + [{"ld_x": 63}, {"ld_u": 63}], "ok"),
    "linearise_batch_dev": (lambda n: [("x", ("f8", 18 * n)), ("ld_x", n), ("u", ("f8", 4 * n)), ("ld_u", n), ("N", n), ("eps", 1e-5),
                                       ("scheme", 0), ("A", ("f8", 324 * n)), ("B", ("f8", 72 * n))] + _sel(n) +
                            [("status", ("i4", n))], ["x", "u", "A", "B"], _LIN_BAD + [{"ld_x": 63}, {"ld_u": 63}], "ok"),
    "trim_batch_dev": (lambda n: [("h", ("f8", n)), ("V", ("f8", n)), ("N", n), ("tol", 1e-10), ("maxiter", 100), ("ux0", None),
                                  ("x_trim", ("f8", 18 * n)), ("ld_x", n), ("info", ("f8", 4 * n)), ("ld_info", n)] + _sel(n) +
                       [("status", ("i4", n))], ["h", "V", "x_trim"], _TRIM_BAD + [{"ld_x": 63}, {"ld_info": 63}], "ok"),
    "state_summary_batch_dev": (lambda n: [("x", ("f8", 18 * n)), ("ld_x", n), ("N", n), ("status", ("i4", n)),
                                           ("row", ("host", "f8", 74))], ["x", "row"], [{"ld_x": 63}], "rows"),
    "step_batch_stats_dev": (lambda n: [("x", ("f8", 18 * n)), ("ld_x", n), ("u", ("f8", 4 * n)), ("ld_u", n), ("N", n), ("K", 4),
                                        ("snap_every", 2), ("dt", 1e-3), ("lqr", None)] + _sel(n) +
                             [("rows", ("host", "f8", 2 * 74)), ("status", ("i4", n))],
                             ["x", "u", "rows", "status"], _SNAP_BAD + [{"ld_x": 63}, {"ld_u": 63}], "rows"),
}


@pytest.mark.parametrize("name", sorted(_ENTRY))
def test_argument_checks(f16, name):
    """Each rejected argument gives F16_ERR_ARG, names the entry point in f16_last_error() and leaves every array as it was.
    N = 0 is F16_OK and touches nothing, except that the statistics calls write their empty rows and the probes reject it."""
    L = f16.lib
    args_of, nulls, bad, empty = _ENTRY[name]
    fn, on_dev, n = getattr(L, name), name.endswith("_dev"), 64
    fill = {"f8": -1.2345678901234567e+300, "i4": 0x5A5A5A5A, "u1": 0xA5}

    def call(**over):
        arrays, vals, laws = {}, [], []
        for k, v in args_of(n):
            v = over.get(k, v)
            if isinstance(v, tuple) and v[0] == "law":
                laws.append(f16.LqrLaw())
                laws[-1].n_sel, laws[-1].sel[0] = v[1], v[2]
                v = ctypes.byref(laws[-1])
            elif isinstance(v, tuple):
                host = v[0] == "host"
                kind, count = v[-2:]
                a = np.full(count, fill[kind], dtype={"f8": np.float64, "i4": np.int32, "u1": np.uint8}[kind])
                p = a.ctypes.data
                if on_dev and not host:
                    p = L.f16_dev_alloc(a.nbytes)
                    assert p and L.f16_memcpy_h2d(p, a.ctypes.data, a.nbytes) == 0
                arrays[k] = (a, p if on_dev and not host else None)
                v = ctypes.cast(ctypes.c_void_p(p), ctypes.POINTER(np.ctypeslib.as_ctypes_type(a.dtype)))
            vals.append(v)
        rc = fn(*vals)
        assert L.f16_sync() == 0
        now = {}
        for k, (a, p) in arrays.items():
            b = a.copy()
            if p is not None:
                assert L.f16_memcpy_d2h(b.ctypes.data, p, b.nbytes) == 0
                L.f16_dev_free(p)
            now[k] = (a, b)
        return rc, now

    rejections = [{k: None} for k in nulls] + [{"N": -1}] + bad
    for over in rejections:
        rc, arrays = call(**over)
        assert rc == -3, (name, over, rc)
        assert name.encode() in L.f16_last_error(), (name, over, L.f16_last_error())
        for k, (a, b) in arrays.items():
            assert np.array_equal(a, b), (name, over, k)
    rc, arrays = call(N=0)
    assert rc == (-3 if empty == "arg" else 0), (name, rc)
    for k, (a, b) in arrays.items():
        if empty == "rows" and k in ("row", "rows"):
            rows = b.reshape(-1, 74)
            assert np.all(rows[:, :2] == 0) and np.all(rows[:, 2:20] == np.inf) and np.all(rows[:, 20:38] == -np.inf), name
        else:
            assert np.array_equal(a, b), (name, k)
