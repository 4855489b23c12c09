"""GPU parity tests: libf16_b200.so (CUDA, through its C ABI) against the oracle and the golden vectors.

Tolerances (BASELINE.json north_star): derivatives <= 1e-12, trajectories <= 1e-9 after 10 s, Jacobians <= 1e-8,
table cells bit-exact.  "Relative" is scaled as SURVEY.md fact 8 prescribes: |a-b| <= tol * max(|ref|, rms of that
output over the batch) -- pure relative error is meaningless for derivatives that cancel to ~0 at trim.
In strict mode the table lookups must be bit-identical to the reference (no transcendental is involved).
"""
import ctypes
import os

import numpy as np
import pytest

from _inputs import X_TRIM_XCG25, X_TRIM_XCG35, perturbed_trim, random_envelope_xu
from conftest import REPO, load_golden, scaled_err
from oracle import HIFI_NAMES, PORT, REF
from oracle import make_lqr as orc_make_lqr

pytestmark = pytest.mark.gpu

TOL_DERIV = 1e-12
TOL_TRAJ = 1e-9
TOL_JAC = 1e-8


def jac_bar(xdot, scheme):
    """Parity bar of a finite-difference Jacobian entry in row i: 1e-8 absolute plus the quotient's own noise floor,
    4 ulp(|f_i|) / h (h = eps forward, 2 eps central; eps = 1e-5).  The reference's OWN source built with -O3 -march=native
    moves the forward A by 2.3e-8 on the 900 ft/s navigation rows (profiles/r02_jacobian_noise_floor.md): one ulp of f
    divided by eps is already 1.1e-8 there.  Wherever |f_i| < 100 the bar is the plain 1e-8.  xdot: [18][N] -> [N][18][1]."""
    h = 1e-5 * (2 if scheme in (1, "central") else 1)
    return TOL_JAC + 4 * np.spacing(np.abs(np.asarray(xdot))).T[:, :, None] / h


def checker(oracle):
    """the reference's own .so when oracle/_ref travelled with the repo, else the pinned C restatement"""
    return REF if oracle.have_ref else PORT


@pytest.fixture(params=["strict", "fast"])
def mode(request, f16):
    prev = f16.lib.f16_set_math_mode(f16.MATH_FAST if request.param == "fast" else f16.MATH_STRICT)
    yield request.param
    f16.lib.f16_set_math_mode(prev)


# ---------------------------------------------------------------------------------------------------------
# the reference's two legacy symbols, called exactly as env.py:100 and utils.py:291 call them
# ---------------------------------------------------------------------------------------------------------
def test_legacy_nlplant_and_atmos(f16, oracle, golden):
    xcg = float(golden["xcg"])
    f16.lib.f16_set_default_xcg(xcg)
    x = golden["nl_xu"].copy()
    for k, fi in enumerate((1, 0)):
        xdot = np.zeros(18)
        f16.lib.Nlplant(ctypes.c_void_p(x[:17].ctypes.data), ctypes.c_void_p(xdot.ctypes.data), ctypes.c_int(fi))
        assert f16.lib.f16_last_status() == 0
        ref = golden["nl_xdot"][k]
        assert np.max(np.abs(xdot - ref) / np.maximum(np.abs(ref), 1e-3)) < TOL_DERIV, (fi, xdot - ref)
    coeff = np.zeros(3)
    f16.lib.atmos(ctypes.c_double(x[2]), ctypes.c_double(x[6]), ctypes.c_void_p(coeff.ctypes.data))
    assert np.allclose(coeff, oracle.atmos(x[2], x[6]), rtol=1e-14, atol=0)
    f16.lib.f16_set_default_xcg(0.25)


def test_atmosphere_over_the_whole_altitude_range(f16, oracle, mode):
    """atmos_batch against the oracle's atmos (the reference's pow(tfac, 4.14), C/nlplant.c:467-490) from -10 000 to 120 000 ft:
    the device build's table-and-series power (f16_model.cuh::pow_4_14) on every one of its 48 centres, half-way between them,
    at both ends of its table, and the libm fall-back beyond.  mach is exact to rounding; qbar and ps carry the power: 4 ulp."""
    c = (18.5 + np.arange(48)) / 64                                   # centres of the table, as tfac
    tf = np.concatenate([c, c + 0.5 / 64, c - 0.5 / 64, np.nextafter(c + 0.5 / 64, 0), [0.28125, np.nextafter(1.03125, 0), 1.03125,
                                                                                        0.2, 1.07]])
    alt = np.concatenate([(1 - tf) / 0.703e-5, np.linspace(-10_000, 120_000, 5001), [0.0, 35000.0, np.nextafter(35000.0, 0), 1e5]])
    vt = np.full(alt.size, 650.0)
    vt[::7] = 0.005
    out = f16.atmos(alt, vt)
    ref = np.array([oracle.atmos(float(a), float(v)) for a, v in zip(alt, vt)]).T
    bar = 4 * np.spacing(np.abs(ref))   # both modes run the parity build here
    assert np.all(np.abs(out - ref) <= bar), float(np.max(np.abs(out - ref) / np.abs(ref)))


def test_dropin_shim_libraries(f16, golden):
    """C/nlplant_xcg25.so and C/nlplant_xcg35.so as parameters.py:108-114 loads them"""
    xcg = float(golden["xcg"])
    name = "nlplant_xcg35.so" if xcg == 0.35 else "nlplant_xcg25.so"
    shim = ctypes.CDLL(os.path.join(REPO, "f16_mpc_oop_py_b200", "dropin", "C", name))
    x = golden["nl_xu"].copy()
    xdot = np.zeros(18)
    shim.Nlplant(ctypes.c_void_p(x.ctypes.data), ctypes.c_void_p(xdot.ctypes.data), ctypes.c_int(1))
    ref = golden["nl_xdot"][0]
    assert np.max(np.abs(xdot - ref) / np.maximum(np.abs(ref), 1e-3)) < TOL_DERIV
    coeff = np.zeros(3)
    shim.atmos(ctypes.c_double(1e4), ctypes.c_double(500.0), ctypes.c_void_p(coeff.ctypes.data))
    assert np.isfinite(coeff).all() and coeff[0] > 0


def test_legacy_out_of_envelope_is_nan_not_a_crash(f16):
    x = load_golden("xcg25")["nl_xu"].copy()
    x[7] = np.deg2rad(45.001)   # the shipped reference .so segfaults here (SURVEY fact 5)
    xdot = np.zeros(18)
    f16.lib.Nlplant(ctypes.c_void_p(x.ctypes.data), ctypes.c_void_p(xdot.ctypes.data), ctypes.c_int(1))
    assert np.isnan(xdot).all() and f16.lib.f16_last_status() == 1 << 18
    f16.lib.Nlplant(ctypes.c_void_p(x.ctypes.data), ctypes.c_void_p(xdot.ctypes.data), ctypes.c_int(0))
    assert np.isfinite(xdot).all()   # lofi extrapolates (lofi_F16_AeroData.c:31-39)
    f16.lib.Nlplant(ctypes.c_void_p(x.ctypes.data), ctypes.c_void_p(xdot.ctypes.data), ctypes.c_int(7))
    assert np.isnan(xdot).all() and f16.lib.f16_last_status() == 1 << 22


# ---------------------------------------------------------------------------------------------------------
# table interpolation: values and cell indices bit-exact (BASELINE cfg 3 stress: every breakpoint, +-1 ulp)
# ---------------------------------------------------------------------------------------------------------
def _probe_points():
    r = np.random.default_rng(5)
    A1 = [-20.0 + 5 * i for i in range(14)]
    B1 = [-30., -25, -20, -15, -10, -8, -6, -4, -2, 0, 2, 4, 6, 8, 10, 15, 20, 25, 30]
    D1 = [-25., -10, 0, 10, 25]
    pts = [(r.uniform(-20, 45), r.uniform(-30, 30), r.uniform(-25, 25)) for _ in range(20000)]
    # a uniform alpha sweep over the whole hifi grid
    pts += [(a, r.uniform(-30, 30), r.uniform(-25, 25)) for a in np.linspace(-20, 45, 2601)]

    def around(v, lo, hi):
        out = [v]
        if v < hi:
            out.append(np.nextafter(v, np.inf))
        if v > lo:
            out.append(np.nextafter(v, -np.inf))
        return out

    for a in A1:
        for aa in around(a, -20, 45):
            for b in B1:
                pts.append((aa, b, float(r.choice(D1))))
            pts.append((aa, r.uniform(-30, 30), r.uniform(-25, 25)))
    for b in B1:
        for bb in around(b, -30, 30):
            pts.append((r.uniform(-20, 45), bb, r.uniform(-25, 25)))
    for d in D1:
        for dd in around(d, -25, 25):
            pts.append((r.uniform(-20, 45), r.uniform(-30, 30), dd))
    return np.array(pts).T.copy()


@pytest.fixture
def strict_mode(f16):
    """strict math for the duration of one test; the previous mode is restored (VERDICT r01 weak #10)"""
    prev = f16.lib.f16_set_math_mode(f16.MATH_STRICT)
    yield
    f16.lib.f16_set_math_mode(prev)


def test_hifi_lookup_bit_exact(f16, oracle, strict_mode):
    a, b, e = _probe_points()
    n = a.size
    coef = np.empty((44, n))
    cells = np.empty((8, n), dtype=np.int32)
    st = np.zeros(n, dtype=np.int32)
    rc = f16.lib.f16_hifi_probe(a.ctypes.data, b.ctypes.data, e.ctypes.data, n, coef.ctypes.data, cells.ctypes.data,
                                st.ctypes.data)
    assert rc == 0 and not st.any()
    ref = np.array([oracle.hifi(a[i], b[i], e[i]) for i in range(n)]).T
    bad = [HIFI_NAMES[i] for i in range(44) if not np.array_equal(coef[i], ref[i])]
    assert not bad, bad
    ref_cells = np.empty((8, n), dtype=np.int32)
    for i in range(n):
        row = []
        for ax, v in (("ALPHA1", a[i]), ("BETA1", b[i]), ("DH1", e[i]), ("DH2", e[i])):
            _, lo, hi = oracle.cell(ax, v)
            row += [lo, hi]
        ref_cells[:, i] = row
    assert np.array_equal(cells, ref_cells)


def test_hifi_lookup_outside_grid_is_flagged(f16):
    a = np.array([45.0001, 60.0, 90.0, -20.0001, 0.0, 0.0, np.nan, 10.0])
    b = np.array([0.0, 0.0, 0.0, 0.0, 30.01, 0.0, 0.0, -31.0])
    e = np.array([0.0, 0.0, 0.0, 0.0, 0.0, 25.5, 0.0, 0.0])
    n = a.size
    coef = np.empty((44, n))
    cells = np.empty((8, n), dtype=np.int32)
    st = np.zeros(n, dtype=np.int32)
    assert f16.lib.f16_hifi_probe(a.ctypes.data, b.ctypes.data, e.ctypes.data, n, coef.ctypes.data, cells.ctypes.data,
                                  st.ctypes.data) == 0
    assert list(st) == [1 << 18] * 4 + [1 << 19, 1 << 20, 1 << 18, 1 << 19]
    assert np.isnan(coef).all()


def test_lofi_lookup(f16, oracle, strict_mode):
    r = np.random.default_rng(4)
    n = 20000
    a = np.concatenate([r.uniform(-20, 90, n - 60), np.arange(-20, 100, 5.0)[:24], np.arange(-20, 100, 5.0)[:24] + 1e-13,
                        np.full(12, 7.5)])
    b = r.uniform(-30, 30, n)
    b[-12:] = [0, 5, 10, 15, 20, 25, 30, -30, -5, 1e-300, -1e-300, 29.999999]
    e = r.uniform(-25, 25, n)
    e[:5] = [-24, -12, 0, 12, 24]
    da, dr = r.uniform(-1, 1, n), r.uniform(-1, 1, n)
    out = np.empty((19, n))
    assert f16.lib.f16_lofi_probe(a.ctypes.data, b.ctypes.data, e.ctypes.data, da.ctypes.data, dr.ctypes.data, n,
                                  out.ctypes.data) == 0
    L = oracle.lib
    ref = np.empty((19, n))
    buf = np.zeros(9)
    p = buf.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    for i in range(n):
        L.orc_lofi_damping(a[i], p); ref[0:9, i] = buf[:9]
        L.orc_lofi_dmomdcon(a[i], b[i], p); ref[9:13, i] = buf[:4]
        L.orc_lofi_clcn(a[i], b[i], p); ref[13:15, i] = buf[:2]
        L.orc_lofi_cxcm(a[i], e[i], p); ref[15:17, i] = buf[:2]
        ref[17, i] = L.orc_lofi_cz(a[i], b[i], e[i])
        ref[18, i] = -.02 * b[i] + .021 * da[i] + .086 * dr[i]
    # bit-exact except cz, whose pow(beta/57.3, 2) is glibc's (about 1 in 5000 arguments is not the rounded product)
    for row in range(17):
        assert np.array_equal(out[row], ref[row]), row
    assert np.max(np.abs(out[17] - ref[17])) < 1e-15
    assert np.allclose(out[18], ref[18], rtol=0, atol=1e-17)


def test_fast_image_and_cell_search_on_the_device(f16, oracle):
    """f16_fast_probe: the F16_MATH_FAST table image with the step kernel's own cell search (csrc/f16_fast.cuh:
    locate_hifi) against getHyperCube (mexndinterp.c:97-143) and the reference aggregators (hifi:1871-1934): random points,
    every breakpoint of ALPHA / BETA1 / DH1 / DH2, +-1 ulp, and the 1e-12 .. 1e-6 bands on both sides (VERDICT r01 #1)."""
    from _probe import check_fast_probe, probe_points
    pts = probe_points()
    n = pts.shape[1]
    a, b, e = (np.ascontiguousarray(pts[i]) for i in range(3))
    coef, cells, lam = np.empty((44, n)), np.empty((4, n), dtype=np.int32), np.empty((4, n))
    st = np.zeros(n, dtype=np.int32)
    assert f16.lib.f16_fast_probe(a.ctypes.data, b.ctypes.data, e.ctypes.data, n, coef.ctypes.data, cells.ctypes.data,
                                  lam.ctypes.data, st.ctypes.data) == 0
    assert not st.any()
    s = check_fast_probe(oracle, pts, coef, cells, lam)
    assert s["worst_coef_err"] < 1e-13, s
    # outside the tables: flagged, NaN, cell -1
    a2, b2, e2 = np.array([45.0001, 0.0, 0.0]), np.array([0.0, -30.5, 0.0]), np.array([0.0, 0.0, 25.5])
    c2, k2, l2, s2 = np.empty((44, 3)), np.empty((4, 3), dtype=np.int32), np.empty((4, 3)), np.zeros(3, dtype=np.int32)
    assert f16.lib.f16_fast_probe(a2.ctypes.data, b2.ctypes.data, e2.ctypes.data, 3, c2.ctypes.data, k2.ctypes.data,
                                  l2.ctypes.data, s2.ctypes.data) == 0
    assert list(s2) == [1 << 18, 1 << 19, 1 << 20] and np.isnan(c2).all() and (k2 == -1).all()


# ---------------------------------------------------------------------------------------------------------
# Nlplant_batch (BASELINE cfg 3: hifi/lofi x xcg 0.25/0.35)
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fi", [1, 0])
@pytest.mark.parametrize("xcg", [0.25, 0.35])
def test_nlplant_batch_parity(f16, oracle, mode, fi, xcg):
    xu = random_envelope_xu(20000, seed=21, hifi=bool(fi))
    ref, rst = oracle.nlplant_batch(xu, fi, xcg, checker(oracle))
    out, st = f16.nlplant(xu, fi, xcg)
    assert not st.any() and not rst.any()
    err = scaled_err(out, ref)
    assert err < TOL_DERIV, err


def test_nlplant_batch_alpha_sweep_and_status(f16, oracle):
    """alpha swept -20..90 deg: hifi has a reference answer on [-20,45] only, lofi everywhere (SURVEY fact 5)"""
    n = 4096
    xu = random_envelope_xu(n, seed=3, hifi=False)
    xu[7] = np.deg2rad(np.linspace(-20, 90, n))
    for fi in (1, 0):
        out, st = f16.nlplant(xu, fi, 0.35)
        ref, rst = oracle.nlplant_batch(xu, fi, 0.35, checker(oracle))
        assert np.array_equal(st, rst)
        ok = st == 0
        if fi == 1:
            deg = np.rad2deg(xu[7]) if False else xu[7] * (180.0 / np.pi)
            assert np.array_equal(ok, deg <= 45.0) and (st[~ok] == 1 << 18).all()
            assert np.isnan(out[:, ~ok]).all()
        else:
            assert ok.all()
        assert scaled_err(out[:, ok], ref[:, ok]) < TOL_DERIV


def test_nlplant_batch_mixed_fidelity_and_xcg(f16, oracle):
    n = 10000
    r = np.random.default_rng(8)
    xu = random_envelope_xu(n, seed=9, hifi=True)
    fi = r.integers(0, 2, n).astype(np.uint8)
    xcg = np.where(r.integers(0, 2, n) == 1, 0.35, 0.25)
    out, st = f16.nlplant(xu, fi, xcg)
    assert not st.any()
    for f in (0, 1):
        for c in (0.25, 0.35):
            m = (fi == f) & (xcg == c)
            ref, _ = oracle.nlplant_batch(np.ascontiguousarray(xu[:, m]), f, c, checker(oracle))
            assert scaled_err(out[:, m], ref) < TOL_DERIV
    fi[5] = 9
    out, st = f16.nlplant(xu, fi, xcg)
    assert st[5] == 1 << 22 and np.isnan(out[:, 5]).all() and not st[6]


@pytest.mark.parametrize("fi", [1, 0])
def test_oneshot_fast_kernels_load_paths_agree(f16, fi):
    """The F16_MATH_FAST one-shot kernels fetch full, 16-byte-aligned tasks of 32 aircraft by TMA bulk copies and everything
    else (odd N / odd plane stride, ragged last task) by plain loads: every path must give the same bits, for
    Nlplant_batch and calc_xdot_batch, with status words, NaN inputs and out-of-table aircraft in the batch."""
    prev = f16.lib.f16_set_math_mode(f16.MATH_FAST)
    try:
        n = 6000
        xu = random_envelope_xu(n, seed=77, hifi=bool(fi))
        r = np.random.default_rng(78)
        x = np.vstack([xu, r.uniform(-30, 30, (1, n))])
        u = np.stack([r.uniform(500, 20000, n), r.uniform(-30, 30, n), r.uniform(-25, 25, n), r.uniform(-35, 35, n)])
        x[7, 5] = np.deg2rad(60.0)      # outside the hifi tables (lofi: fine)
        x[8, 6] = np.deg2rad(-31.0)     # outside both
        x[9, 7] = np.nan                # NaN in a rate: reference-order path, NaN derivatives, status 0
        x[2, 8] = 120000.0              # altitude beyond the density table of the fast arithmetic (tfac = 0.156)
        x[4, 9] = 4.0e9                 # Euler angle beyond 2^30
        fb = f16.F16Batch(x, u, fi_flag=fi, xcg=0.3)
        full = fb._calc_xdot(x, u)
        full_st = fb.last_status.copy()
        nl, nl_st = f16.nlplant(x[:17], fi, 0.3)
        assert full_st[6] == 1 << 19 and (full_st[5] == (1 << 18 if fi else 0)) and full_st[7] == 0 and np.isnan(full[9:12, 7]).all()
        assert np.isfinite(full[:, 8]).all() and np.isfinite(full[:, 9]).all() and np.isfinite(full[:, 10:]).all()
        for m in (4096, 4098, 4099, 4127, 5001):
            fbm = f16.F16Batch(x[:, :m], u[:, :m], fi_flag=fi, xcg=0.3)
            out = fbm._calc_xdot(np.ascontiguousarray(x[:, :m]), np.ascontiguousarray(u[:, :m]))
            assert np.array_equal(out, full[:, :m], equal_nan=True), m
            assert np.array_equal(fbm.last_status, full_st[:m]), m
            o2, s2 = f16.nlplant(np.ascontiguousarray(x[:17, :m]), fi, 0.3)
            assert np.array_equal(o2, nl[:, :m], equal_nan=True) and np.array_equal(s2, nl_st[:m]), m
        # the small-batch path (tables through L2) is the parity build: the bits and status words of F16_MATH_STRICT
        xs, us = np.ascontiguousarray(x[:, :1000]), np.ascontiguousarray(u[:, :1000])
        fbs = f16.F16Batch(xs, us, fi_flag=fi, xcg=0.3)
        small = fbs._calc_xdot(xs, us)
        small_st = fbs.last_status.copy()
        fin = np.isfinite(full[:, :1000]).all(axis=0) & (full_st[:1000] == 0)
        assert scaled_err(small[:, fin], full[:, :1000][:, fin]) < TOL_DERIV
        f16.lib.f16_set_math_mode(f16.MATH_STRICT)
        assert np.array_equal(small, fbs._calc_xdot(xs, us), equal_nan=True) and np.array_equal(small_st, fbs.last_status)
    finally:
        f16.lib.f16_set_math_mode(prev)


def test_fast_mode_off_its_kernels_is_the_parity_build(f16):
    """F16_MATH_FAST runs f16_fast.cuh only where its kernels are taken (include/f16_b200.h): one-shot batches below 4096
    aircraft, anything with table staging off, the legacy symbols, atmos_batch and the table probes give the bits and status
    words of F16_MATH_STRICT -- a result does not depend on the batch size through a third arithmetic.  A fast-mode trim runs
    f16_fast.cuh at every batch size: a few points get the bits they get inside a batch of 1024."""
    r = np.random.default_rng(31)
    batches = []
    for n in (1, 31, 1000, 4095):
        xu = random_envelope_xu(n, seed=n, hifi=True)
        x = np.vstack([xu, r.uniform(-30, 30, (1, n))])
        u = np.stack([r.uniform(500, 20000, n), r.uniform(-30, 30, n), r.uniform(-25, 25, n), r.uniform(-35, 35, n)])
        if n > 1:
            x[7, n - 1] = np.deg2rad(60.0)   # outside the hifi tables: a status word
        fi, xcg = r.integers(0, 2, n).astype(np.uint8), r.uniform(0.25, 0.35, n)
        batches.append((x, u, [(1, 0.3), (0, 0.3), (fi, xcg)]))
    nl = load_golden("xcg25")["nl_xu"].copy()
    alt = np.linspace(-10_000, 120_000, 3001)
    vt = np.linspace(0.005, 1000.0, alt.size)
    a, b, e = _probe_points()
    m = a.size
    da, dr = r.uniform(-1, 1, m), r.uniform(-1, 1, m)
    h, v = np.array([5000.0, 20000.0, 35000.0]), np.array([400.0, 700.0, 900.0])
    xb = np.vstack([random_envelope_xu(5000, seed=5, hifi=True), r.uniform(-30, 30, (1, 5000))])
    ub = np.stack([r.uniform(500, 20000, 5000), r.uniform(-30, 30, 5000), r.uniform(-25, 25, 5000), r.uniform(-35, 35, 5000)])

    def run():
        out = []
        for x, u, sels in batches:
            for fi, xcg in sels:
                out += list(f16.nlplant(x[:17], fi, xcg))
                fb = f16.F16Batch(x, u, fi_flag=fi, xcg=xcg)
                out += [fb._calc_xdot(x, u), fb.last_status.copy()]
        for fi in (1, 0):
            xd = np.zeros(18)
            f16.lib.Nlplant(ctypes.c_void_p(nl.ctypes.data), ctypes.c_void_p(xd.ctypes.data), ctypes.c_int(fi))
            out += [xd, f16.lib.f16_last_status()]
        coeff = np.zeros(3)
        f16.lib.atmos(ctypes.c_double(nl[2]), ctypes.c_double(nl[6]), ctypes.c_void_p(coeff.ctypes.data))
        out += [coeff, f16.atmos(alt, vt)]
        coef, cells, st = np.empty((44, m)), np.empty((8, m), dtype=np.int32), np.zeros(m, dtype=np.int32)
        assert f16.lib.f16_hifi_probe(a.ctypes.data, b.ctypes.data, e.ctypes.data, m, coef.ctypes.data, cells.ctypes.data,
                                      st.ctypes.data) == 0
        lofi = np.empty((19, m))
        assert f16.lib.f16_lofi_probe(a.ctypes.data, b.ctypes.data, e.ctypes.data, da.ctypes.data, dr.ctypes.data, m,
                                      lofi.ctypes.data) == 0
        out += [coef, cells, st, lofi]
        prev = f16.lib.f16_set_table_staging(0)
        try:
            fb = f16.F16Batch(xb, ub, fi_flag=1, xcg=0.3)
            out += [fb._calc_xdot(xb, ub), fb.last_status.copy()]
            xt, opt = f16.trim(h[:1], v[:1], fi=1, xcg=0.3)
            out += [xt, opt["fun"], opt["nit"], opt["status"]]
        finally:
            f16.lib.f16_set_table_staging(prev)
        return out

    res = {}
    for mode in (f16.MATH_STRICT, f16.MATH_FAST):
        prev = f16.lib.f16_set_math_mode(mode)
        try:
            res[mode] = run()
        finally:
            f16.lib.f16_set_math_mode(prev)
    differ = [i for i, (s, q) in enumerate(zip(res[f16.MATH_STRICT], res[f16.MATH_FAST])) if not np.array_equal(s, q, equal_nan=True)]
    assert not differ, differ
    prev = f16.lib.f16_set_math_mode(f16.MATH_FAST)
    try:
        hb, vb = np.resize(h, 1024), np.resize(v, 1024)
        for fi in (1, 0):
            few, big = f16.trim(h, v, fi=fi, xcg=0.3), f16.trim(hb, vb, fi=fi, xcg=0.3)
            assert np.array_equal(few[0], big[0][:, :3], equal_nan=True), fi
            assert all(np.array_equal(few[1][k], big[1][k][:3], equal_nan=True) for k in few[1]), fi
    finally:
        f16.lib.f16_set_math_mode(prev)


def test_nlplant_batch_edges(f16):
    out, st = f16.nlplant(np.zeros((17, 0)))
    assert out.shape == (18, 0)
    xu = random_envelope_xu(1, seed=1)
    out1, _ = f16.nlplant(xu)
    big = np.repeat(xu, 70001, axis=1)          # ragged: not a multiple of any CTA size
    outb, _ = f16.nlplant(big)
    assert np.array_equal(outb, np.repeat(out1, 70001, axis=1))   # same input -> same bits in every lane/CTA
    assert f16.lib.Nlplant_batch(None, None, None, 1, None, 0.25, 5, None) == -3   # F16_ERR_ARG


# ---------------------------------------------------------------------------------------------------------
# _calc_xdot: actuators + LEF + Nlplant (env.py:65-103)
# ---------------------------------------------------------------------------------------------------------
def test_calc_xdot_matches_env_py_golden(f16, mode, golden):
    fb = f16.F16Batch(golden["xs"].T, golden["us"].T, fi_flag=int(golden["fi"]), xcg=float(golden["xcg"]))
    xd = fb._calc_xdot(golden["xs"].T, golden["us"].T)
    assert not fb.last_status.any()
    assert scaled_err(xd, golden["xdots"].T) < TOL_DERIV


def test_actuator_limits_like_the_reference_tests(f16):
    """test_env.py:40-147 restated: command saturation and rate limits of the actuator models"""
    g = load_golden("xcg25")
    x, u = g["x_trim"].copy(), g["u_trim"].copy()
    fb = f16.F16Batch(x, u)
    for idx, (lo, hi, rate) in zip((13, 14, 15), ((-25, 25, 60), (-21.5, 21.5, 80), (-30, 30, 120))):
        xs = np.repeat(x[:, None], 4, axis=1)
        us = np.repeat(u[:, None], 4, axis=1)
        xs[idx, 0], us[idx - 12, 0] = hi, hi + 10      # at the upper limit, demanding more: no motion
        xs[idx, 1], us[idx - 12, 1] = lo, lo - 10
        xs[idx, 2], us[idx - 12, 2] = 0.0, hi           # far away: rate limited
        xs[idx, 3], us[idx - 12, 3] = 0.0, lo
        xd = fb._calc_xdot(xs, us)
        assert xd[idx, 0] == 0 and xd[idx, 1] == 0 and xd[idx, 2] == rate and xd[idx, 3] == -rate
    xs = np.repeat(x[:, None], 2, axis=1)
    us = np.repeat(u[:, None], 2, axis=1)
    xs[12, 0], us[0, 0] = 19000, 30000
    xs[12, 1], us[0, 1] = 1000, 19000
    xd = fb._calc_xdot(xs, us)
    assert xd[12, 0] == 0 and xd[12, 1] == 10000


# ---------------------------------------------------------------------------------------------------------
# step_batch: fused Euler steps (env.py:105-130)
# ---------------------------------------------------------------------------------------------------------
def test_cfg1_single_aircraft_10s_open_loop(f16, oracle, mode):
    """BASELINE cfg 1: one hifi F-16, xcg 0.35, trim at 10000 ft / 700 ft/s, dt = 0.001 for 10 s"""
    g = load_golden("xcg35")
    fb = f16.F16Batch(g["x_trim"], g["u_trim"], fi_flag=1, xcg=0.35)
    fb.step(K=2000)
    assert fb.status[0] == 0 and fb.steps_done[0] == 2000
    assert scaled_err(fb.x[:, 0], g["traj_x"][4]) < TOL_TRAJ      # the real F16.step, 2000 calls
    fb.step(K=8000)
    ref, st = oracle.step_batch(g["x_trim"][:, None].copy(), g["u_trim"][:, None].copy(), 10000, 0.001, 1, 0.35, None,
                                checker(oracle))
    assert st[0] == 0 and fb.status[0] == 0
    rel = np.abs(fb.x[:, 0] - ref[:, 0]) / np.maximum(np.abs(ref[:, 0]), 1e-3)
    assert rel.max() < TOL_TRAJ, rel
    # SURVEY 8c known answer 3
    assert abs(fb.x[0, 0] - 7000.002274) < 1e-5 and abs(fb.x[2, 0] - 9999.939040) < 1e-5


@pytest.mark.parametrize("tag", ["xcg25", "xcg35", "lofi_xcg25"])
def test_step_batch_perturbed_trim(f16, oracle, mode, tag):
    """BASELINE cfg 2 at a size the oracle finishes in seconds: +-5 % about trim, 2 s of flight"""
    g = load_golden(tag)
    fi, xcg = int(g["fi"]), float(g["xcg"])
    x, u = perturbed_trim(512, g["x_trim"])
    ref, rst = oracle.step_batch(x, u, 2000, 0.001, fi, xcg, None, checker(oracle))
    fb = f16.F16Batch(x, u, fi_flag=fi, xcg=xcg)
    fb.step(K=2000)
    alive = (rst == 0) & (fb.status == 0)
    assert alive.mean() > 0.5
    # An aircraft that crosses a bound within rounding of step 2000 may be stopped by one implementation and not (yet) by
    # the other: at most one such grazing case in 512 is accepted (none has been observed); everything else must carry the
    # oracle's status word.
    assert int((rst != fb.status).sum()) <= 1, np.flatnonzero(rst != fb.status)
    assert scaled_err(fb.x[:, alive], ref[:, alive]) < TOL_TRAJ
    frozen = (rst != 0) & (fb.status == rst)
    if frozen.any():
        assert scaled_err(fb.x[:, frozen], ref[:, frozen]) < 1e-6


def test_step_restartable_and_device_api(f16):
    """K = a then K = b is bit-identical to K = a + b; the _dev entry point equals the host one"""
    g = load_golden("xcg25")
    x, u = perturbed_trim(100_000, g["x_trim"], seed=5)
    a = f16.F16Batch(x, u)
    a.step(K=30)
    a.step(K=70)
    b = f16.F16Batch(x, u)
    b.step(K=100)
    assert np.array_equal(a.x, b.x) and np.array_equal(a.status, b.status)
    n = x.shape[1]
    L = f16.lib
    dx, du = L.f16_dev_alloc(x.nbytes), L.f16_dev_alloc(u.nbytes)
    dst = L.f16_dev_alloc(4 * n)
    assert dx and du and dst
    assert L.f16_memcpy_h2d(dx, x.ctypes.data, x.nbytes) == 0 and L.f16_memcpy_h2d(du, u.ctypes.data, u.nbytes) == 0
    before = L.f16_launch_count()
    assert L.step_batch_dev(dx, n, du, n, n, 100, 0.001, None, None, 1, None, 0.25, dst, None) == 0
    assert L.f16_sync() == 0 and L.f16_launch_count() == before + 1
    out = np.empty_like(x)
    assert L.f16_memcpy_d2h(out.ctypes.data, dx, x.nbytes) == 0
    for p in (dx, du, dst):
        L.f16_dev_free(p)
    assert np.array_equal(out, b.x)


def test_step_staged_tables_equal_l2_tables(f16, mode):
    """tables staged in shared memory by TMA (384 threads per CTA) == tables read through L2 (256 threads per CTA), in both
    math modes: the fast kernel has its own table image and instantiations"""
    g = load_golden("xcg35")
    x, u = perturbed_trim(20_000, g["x_trim"], seed=6)
    outs = []
    for staging in (1, 0):
        f16.lib.f16_set_table_staging(staging)
        fb = f16.F16Batch(x, u, xcg=0.35)
        fb.step(K=50)
        outs.append(fb.x.copy())
    f16.lib.f16_set_table_staging(1)
    assert np.array_equal(outs[1], outs[0])


@pytest.mark.parametrize("with_law", [False, True])
def test_step_time_chunked_schedule_equals_the_plain_kernel(f16, with_law):
    """F16_MATH_FAST hifi step: long runs are scheduled as (chunk of steps, group of 32 aircraft) items handed between
    warps through global memory (no grid tail).  Same bits as one warp-task per group for all K steps: states, status
    words and steps_done, with aircraft that leave the envelope at different times (xcg 0.35 open loop) and a ragged N."""
    prev_mode = f16.lib.f16_set_math_mode(f16.MATH_FAST)
    try:
        g = load_golden("xcg35")
        n = 120_000 + 17
        x, u = perturbed_trim(n, g["x_trim"], seed=3)
        x[9, 5] = np.nan
        u[1, 6] = np.nan
        x[2, 7] = 99999.9       # leaves the altitude bound within a few steps
        # 400 aircraft at full thrust just below the 900 ft/s bound: they cross it at different steps, i.e. in different chunks
        x[6, 100:500] = np.linspace(880.0, 899.99, 400)
        x[12, 100:500] = 19000.0
        u[0, 100:500] = 19000.0
        law = None
        if with_law:
            sel = list(g["mpc_x_idx"])
            law = f16.make_lqr(-g["K_lqr"], sel, g["x_trim"][sel], g["u_trim"], rows=[1, 2, 3])
        out = {}
        for on in (0, 1):
            prev = f16.lib.f16_set_step_chunking(on)
            fb = f16.F16Batch(x, u, xcg=0.35)
            fb.step(K=1500, lqr=law)
            out[on] = (fb.x.copy(), fb.status.copy(), fb.steps_done.copy())
            f16.lib.f16_set_step_chunking(prev)
        assert np.array_equal(out[0][1], out[1][1]) and np.array_equal(out[0][2], out[1][2])
        assert np.array_equal(out[0][0], out[1][0], equal_nan=True)
        st, done = out[1][1], out[1][2]
        assert (st != 0).sum() > 100 and (st == 0).mean() > 0.5 and np.all(done[st == 0] == 1500) and np.all(done[st != 0] < 1500)
        assert len(np.unique(done[st != 0] // 94)) > 3      # casualties spread over several chunks (chunk = 94 steps)
    finally:
        f16.lib.f16_set_math_mode(prev_mode)


@pytest.mark.parametrize("K", [1, 3, 7])
def test_short_step_tiled_kernel_equals_the_plain_kernel(f16, K):
    """step_batch with K < 8 on >= 4096 aircraft takes the TMA-tiled short-step kernel (f16_step_fast.cu::step_tiled_fast_kernel);
    the same aircraft inside a batch of 4095 take the plain step kernel.  Same bits -- hifi, lofi, a mixed batch with
    per-aircraft xcg, open and closed loop, a ragged batch size, aircraft outside the envelope among them."""
    prev = f16.lib.f16_set_math_mode(f16.MATH_FAST)
    try:
        g = load_golden("xcg35")
        n, m = 70_001, 4095
        x, u = perturbed_trim(n, g["x_trim"], seed=21, frac=0.05)
        x[7, 5::97] = 1.2          # alpha outside the hifi table: stopped with a status word
        x[6, 7::101] = 950.0       # airspeed beyond its bound
        r = np.random.default_rng(2)
        fi_mixed = (r.uniform(size=n) < 0.6).astype(np.uint8)
        xcg_mixed = np.where(r.uniform(size=n) < 0.5, 0.25, 0.35)
        mpc_idx = list(g["mpc_x_idx"])
        law = f16.make_lqr(-g["K_lqr"], mpc_idx, g["x_trim"][mpc_idx], g["u_trim"], rows=[1, 2, 3])
        for fi, xcg in ((1, 0.35), (0, 0.25), (fi_mixed, xcg_mixed)):
            for lqr in (None, law):
                big = f16.F16Batch(x, u, fi_flag=fi, xcg=xcg)
                big.step(K=K, lqr=lqr)
                small = f16.F16Batch(x[:, :m], u[:, :m], fi_flag=fi if np.ndim(fi) == 0 else fi[:m],
                                     xcg=xcg if np.ndim(xcg) == 0 else xcg[:m])
                small.step(K=K, lqr=lqr)
                assert np.array_equal(big.x[:, :m], small.x, equal_nan=True)
                assert np.array_equal(big.status[:m], small.status) and np.array_equal(big.steps_done[:m], small.steps_done)
                assert (big.status != 0).sum() > 100 and (big.status == 0).sum() > 60_000
    finally:
        f16.lib.f16_set_math_mode(prev)


def test_step_freeze_policy(f16, oracle):
    g = load_golden("xcg35")
    x = np.repeat(g["x_trim"][:, None], 6, axis=1)
    u = np.repeat(g["u_trim"][:, None], 6, axis=1)
    x[7, 1] = np.deg2rad(50)
    x[2, 2] = -5.0
    x[9, 3] = np.nan
    u[1, 4] = np.nan
    x[6, 5] = 950.0
    fb = f16.F16Batch(x, u, xcg=0.35)
    fb.step(K=10)
    ref, rst = oracle.step_batch(x, u, 10, 0.001, 1, 0.35)
    assert np.array_equal(fb.status, rst)
    assert list(fb.steps_done) == [10, 0, 0, 0, 0, 0]
    assert np.array_equal(fb.x[:, 1:], x[:, 1:], equal_nan=True)


def test_closed_loop_lqr_fused(f16, oracle, mode):
    """BASELINE cfg 5 at test size: u = u0 - K(x - x_ref) on the mpc states fused into the step"""
    g = load_golden("xcg35")
    r = np.random.default_rng(9)
    sel = list(g["mpc_x_idx"])
    K = np.zeros((3, 9))
    K[0, [2, 5]] = [-30.0, -8.0]      # elevator <- alpha, q: a stabilising pitch damper for the unstable xcg 0.35
    K[1, [0, 4]] = [-3.0, -1.5]       # aileron  <- phi, p
    K[2, [3, 6]] = [2.0, -1.0]        # rudder   <- beta, r
    law = f16.make_lqr(K, sel, g["x_trim"][sel], g["u_trim"], rows=[1, 2, 3])
    olaw = orc_make_lqr(K, sel, g["x_trim"][sel], g["u_trim"], rows=[1, 2, 3])
    x, u = perturbed_trim(256, g["x_trim"], seed=12, frac=0.02)
    ref, rst = oracle.step_batch(x, u, 2000, 0.001, 1, 0.35, olaw, checker(oracle))
    fb = f16.F16Batch(x, u, xcg=0.35)
    fb.step(K=2000, lqr=law)
    alive = (rst == 0) & (fb.status == 0)
    assert alive.mean() > 0.9
    assert scaled_err(fb.x[:, alive], ref[:, alive]) < TOL_TRAJ


def test_lofi_step_over_the_whole_lofi_envelope(f16, oracle, mode):
    """the lofi step (its own kernel on the fast arithmetic in F16_MATH_FAST) from states anywhere in the lofi envelope --
    alpha -20..89 deg (linear extrapolation of the 5-degree grid beyond -10..45), beta to +-29.9 deg either sign, every
    elevator cell, both xcg -- open loop and with a fused feedback law; short horizon so that nobody leaves on the way"""
    from _inputs import random_envelope_xu
    n = 4096
    xu = random_envelope_xu(n, seed=41, hifi=False)
    r = np.random.default_rng(42)
    x = np.vstack([xu, r.uniform(-20, 5, (1, n))])          # lf1
    x[2] = r.uniform(1000, 39000, n)
    x[7, :8] = np.deg2rad([-20.0, -10.0, 0.0, 45.0, 60.0, 89.0, 5.0, -5.0])      # grid nodes and ends
    x[8, 8:14] = np.deg2rad([0.0, 5.0, -5.0, 29.9, -29.9, 15.0])
    x[13, 14:20] = [-25.0, -24.0, -12.0, 0.0, 12.0, 25.0]
    u = np.vstack([r.uniform(1000, 19000, n), r.uniform(-25, 25, n), r.uniform(-21.5, 21.5, n), r.uniform(-30, 30, n)])
    g = load_golden("lofi_xcg25")
    sel = list(g["mpc_x_idx"])
    K = np.zeros((3, 9))
    K[0, [2, 5]] = [-3.0, -0.8]
    K[1, [0, 4]] = [-0.3, -0.15]
    K[2, [3, 6]] = [0.2, -0.1]
    for xcg in (0.25, 0.35):
        for law, olaw in ((None, None), (f16.make_lqr(K, sel, g["x_trim"][sel], g["u_trim"], rows=[1, 2, 3]),
                                         orc_make_lqr(K, sel, g["x_trim"][sel], g["u_trim"], rows=[1, 2, 3]))):
            ref, rst = oracle.step_batch(x, u, 50, 0.001, 0, xcg, olaw, checker(oracle))
            fb = f16.F16Batch(x, u, fi_flag=0, xcg=xcg)
            fb.step(K=50, lqr=law)
            alive = (rst == 0) & (fb.status == 0)
            assert alive.mean() > 0.9 and np.mean(rst != fb.status) < 0.005
            assert scaled_err(fb.x[:, alive], ref[:, alive]) < TOL_TRAJ


def test_step_mixed_fidelity_batch_equals_separate_batches(f16, mode):
    """BASELINE cfg 3 as a step: per-aircraft fidelity flags and xcg in ONE call = the hifi and lofi batches run apart"""
    g = load_golden("xcg25")
    n = 1500
    x, u = perturbed_trim(n, g["x_trim"], seed=77, frac=0.04)
    fi = (np.arange(n) % 3 != 0).astype(np.uint8)
    xcg = np.where(np.arange(n) % 2 == 0, 0.25, 0.35)
    mixed = f16.F16Batch(x, u, fi_flag=fi, xcg=xcg)
    mixed.step(K=300)
    for f in (0, 1):
        m = fi == f
        part = f16.F16Batch(x[:, m], u[:, m], fi_flag=f, xcg=xcg[m])
        part.step(K=300)
        assert np.array_equal(mixed.x[:, m], part.x, equal_nan=True) and np.array_equal(mixed.status[m], part.status)


@pytest.mark.parametrize("with_law", [False, True])
def test_step_large_mixed_batch_is_partitioned_by_fidelity(f16, mode, with_law):
    """a mixed batch big enough for the fidelity partition (f16_partition.cu: stable three-way partition, gather, two
    launches on contiguous ranges, scatter): same bits as the two fidelities run apart, whatever the interleaving;
    aircraft with an invalid flag keep their state and report F16_ST_FIDELITY"""
    g = load_golden("xcg25")
    n = 20000 + 37
    x, u = perturbed_trim(n, g["x_trim"], seed=78, frac=0.04)
    r = np.random.default_rng(5)
    fi = (r.uniform(size=n) < 0.6).astype(np.uint8)
    fi[[3, 4097, n - 1]] = 7                                    # neither model
    xcg = np.where(r.uniform(size=n) < 0.5, 0.25, 0.35)
    law = None
    if with_law:
        sel = list(g["mpc_x_idx"])
        K = np.zeros((3, 9))
        K[0, [2, 5]] = [-3.0, -0.8]
        law = f16.make_lqr(K, sel, g["x_trim"][sel], g["u_trim"], rows=[1, 2, 3])
    mixed = f16.F16Batch(x, u, fi_flag=fi, xcg=xcg)
    mixed.step(K=60, lqr=law)
    for f in (0, 1):
        m = fi == f
        part = f16.F16Batch(x[:, m], u[:, m], fi_flag=f, xcg=xcg[m])
        part.step(K=60, lqr=law)
        assert np.array_equal(mixed.x[:, m], part.x, equal_nan=True) and np.array_equal(mixed.status[m], part.status)
        assert np.array_equal(mixed.steps_done[m], part.steps_done)
    bad = fi == 7
    assert np.all(mixed.status[bad] == 1 << 22) and np.all(mixed.steps_done[bad] == 0) and np.array_equal(mixed.x[:, bad], x[:, bad])


# ---------------------------------------------------------------------------------------------------------
# linearise_batch (env.py:294-342; BASELINE cfg 4)
# ---------------------------------------------------------------------------------------------------------
def test_linearise_matches_env_py_golden(f16, mode, golden):
    """F16.linearise at the trim point of the unmodified reference.  strict: 1e-8 on every entry; fast (the quotient on the
    re-associated arithmetic): 1e-8 everywhere except the two navigation rows, which get the noise-floor bar of jac_bar()."""
    fb = f16.F16Batch(golden["x_trim"], golden["u_trim"], fi_flag=int(golden["fi"]), xcg=float(golden["xcg"]))
    A, B, C, D = fb.linearise(golden["x_trim"], golden["u_trim"], scheme="forward")
    eA, eB = np.abs(A[0] - golden["Ac"]), np.abs(B[0] - golden["Bc"])
    if mode == "strict":
        assert eA.max() < TOL_JAC and eB.max() < TOL_JAC
    else:
        bar = jac_bar(golden["xdot_trim"][:, None], "forward")[0]
        assert (eA <= bar).all() and eB.max() < TOL_JAC and eA[2:].max() < TOL_JAC, (eA.max(), eA[2:].max())
    assert C.shape == (10, 18) and D.shape == (10, 4) and C.sum() == 10


@pytest.fixture(params=[(0, 0), (1, 1)], ids=["strict", "fast_variant1"])
def reference_order_linearise(request, f16):
    """the reference-order Jacobian kernel, reached by default in F16_MATH_STRICT and through f16_set_linearise_variant(1)
    in F16_MATH_FAST"""
    math_mode, variant = request.param
    prev_mode = f16.lib.f16_set_math_mode(f16.MATH_FAST if math_mode else f16.MATH_STRICT)
    prev = f16.lib.f16_set_linearise_variant(variant)
    yield request.param
    f16.lib.f16_set_linearise_variant(prev)
    f16.lib.f16_set_math_mode(prev_mode)


def test_linearise_strict_equals_host_finite_differences(f16):
    """The strict linearise_batch (stages of f shared between the columns, calc_xdot_col) gives the bits of finite
    differences formed on the host from full strict calc_xdot_batch evaluations: the perturbed points built as the kernel
    builds them (x0 + where(i == c, +-eps, 0.0); the forward base point x0 + 0.0, which turns -0.0 into +0.0), IEEE
    quotients, a column NaN wherever one of its evaluations (forward: or the base point's) failed, and the status word the
    OR over every evaluation."""
    g = load_golden("xcg25")
    x, u = perturbed_trim(1000 + 7, g["x_trim"], seed=5, frac=0.04)
    x[13, 5] = 25.0 - 1e-6      # elevator + eps leaves the hifi tables: column 13 of aircraft 5 is NaN
    n = x.shape[1]
    fi = np.ones(n, dtype=np.uint8)
    fi[::3] = 0
    eps = 1e-5
    xu0 = np.vstack([x, u])     # columns 0..17 states, 18..21 inputs
    idx = np.arange(22)[:, None]
    prev = f16.lib.f16_set_math_mode(f16.MATH_STRICT)
    try:
        for scheme in ("forward", "central"):
            signs = (1.0,) if scheme == "forward" else (1.0, -1.0)
            pts = [xu0 + np.where(idx == c, s * eps, 0.0) for s in signs for c in range(22)]
            if scheme == "forward":
                pts.append(xu0 + 0.0)
            xu = np.ascontiguousarray(np.hstack(pts))
            m = len(pts)
            ev = f16.F16Batch(xu[:18], xu[18:], fi_flag=np.tile(fi, m), xcg=0.25)
            f = ev._calc_xdot(xu[:18], xu[18:]).reshape(18, m, n)
            st = ev.last_status.reshape(m, n)
            # forward: f(x0 + eps e_c) - f(x0 + 0.0); central: f(x0 + eps e_c) - f(x0 - eps e_c)
            num = f[:, :22] - f[:, 22:]
            bad = (st[:22] != 0) | (st[22:] != 0)
            q = np.where(bad[None], np.nan, num / (eps if scheme == "forward" else 2 * eps))   # [row][column][aircraft]
            status = np.bitwise_or.reduce(st, axis=0)
            fb = f16.F16Batch(x, u, fi_flag=fi, xcg=0.25)
            A, B, _, _ = fb.linearise(x, u, scheme=scheme, eps=eps)
            assert np.array_equal(fb.last_status, status), scheme
            assert np.array_equal(A, q[:, :18].transpose(2, 0, 1), equal_nan=True), scheme
            assert np.array_equal(B, q[:, 18:].transpose(2, 0, 1), equal_nan=True), scheme
            assert np.isnan(A[5, :, 13]).all() and fb.last_status[5] != 0
    finally:
        f16.lib.f16_set_math_mode(prev)


@pytest.mark.parametrize("scheme", ["forward", "central"])
@pytest.mark.parametrize("fi", [1, 0])
def test_linearise_batch_grid(f16, oracle, scheme, fi, reference_order_linearise):
    """a 16 x 16 altitude x velocity grid about perturbed trims (cfg 4 is 64 x 64; same code path)"""
    g = load_golden("xcg25")
    n = 256 + 13     # ragged last CTA
    x, u = perturbed_trim(n, g["x_trim"], seed=21, frac=0.03)
    x[2] = np.tile(np.linspace(5000, 40000, 16), 17)[:n]
    x[6] = np.repeat(np.linspace(300, 900, 17), 16)[:n]
    sch = 0 if scheme == "forward" else 1
    Ar, Br, rst = oracle.linearise_batch(x, u, 1e-5, sch, fi, 0.25, checker(oracle))
    fb = f16.F16Batch(x, u, fi_flag=fi, xcg=0.25)
    A, B, _, _ = fb.linearise(x, u, scheme=scheme)
    assert np.array_equal(fb.last_status, rst)
    ok = rst == 0
    assert ok.mean() > 0.9
    assert np.abs(A[ok] - Ar[ok]).max() < TOL_JAC and np.abs(B[ok] - Br[ok]).max() < TOL_JAC


@pytest.mark.parametrize("scheme", ["forward", "central"])
@pytest.mark.parametrize("fi", [1, 0])
def test_linearise_fast_kernel_grid(f16, oracle, scheme, fi):
    """F16_MATH_FAST linearise_batch (csrc/f16_linearise_fast.cu: two aircraft per warp on the fast arithmetic) on the same
    16 x 16 altitude x velocity grid: status words equal, rows 2..17 within 1e-8, the two navigation rows within jac_bar()."""
    prev = f16.lib.f16_set_math_mode(f16.MATH_FAST)
    try:
        g = load_golden("xcg25")
        n = 256 + 13     # odd: the last warp-task holds one aircraft
        x, u = perturbed_trim(n, g["x_trim"], seed=21, frac=0.03)
        x[2] = np.tile(np.linspace(5000, 40000, 16), 17)[:n]
        x[6] = np.repeat(np.linspace(300, 900, 17), 16)[:n]
        sch = 0 if scheme == "forward" else 1
        Ar, Br, rst = oracle.linearise_batch(x, u, 1e-5, sch, fi, 0.25, checker(oracle))
        fb = f16.F16Batch(x, u, fi_flag=fi, xcg=0.25)
        A, B, _, _ = fb.linearise(x, u, scheme=scheme)
        assert np.array_equal(fb.last_status, rst)
        ok = rst == 0
        assert ok.mean() > 0.9
        xd = fb._calc_xdot(x, u)
        bar = jac_bar(xd, sch)[ok]
        eA, eB = np.abs(A[ok] - Ar[ok]), np.abs(B[ok] - Br[ok])
        assert (eA <= bar).all() and eB.max() < TOL_JAC and eA[:, 2:].max() < TOL_JAC, (eA.max(), eA[:, 2:].max(), eB.max())
    finally:
        f16.lib.f16_set_math_mode(prev)


def test_linearise_fast_kernel_edge_semantics_equal_the_strict_kernel(f16):
    """Everything that is not an ordinary in-envelope aircraft must come out of the fast-mode kernel exactly as it comes out
    of the strict one (those aircraft are redone on the reference-order arithmetic): columns that leave the tables, a base
    point outside the tables, NaN states / inputs, an altitude beyond the fast density table, huge Euler angles, bad and
    mixed fidelity flags, per-aircraft xcg, N = 1 and odd N."""
    g = load_golden("xcg25")
    n = 777
    x, u = perturbed_trim(n, g["x_trim"], seed=9, frac=0.04)
    x[13, 1] = 25.0 - 1e-6               # elevator + eps leaves DH1: NaN column 13, status DELE
    x[7, 2] = np.deg2rad(45.0) - 2e-6    # alpha + eps leaves the hifi tables
    x[8, 3] = np.deg2rad(31.0)           # base point outside: everything NaN
    x[9, 4] = np.nan
    u[2, 5] = np.nan
    x[17, 6] = np.nan
    x[2, 7] = 120000.0                   # outside the density table of the fast arithmetic
    x[5, 8] = 5.0e9                      # Euler angle beyond 2^30 rad
    x[6, 9] = 0.005                      # below the vt clamp of nlplant.c:104
    fi = np.ones(n, dtype=np.uint8)
    fi[::3] = 0
    fi[10] = 7
    xcg = np.where(np.arange(n) % 2 == 0, 0.25, 0.35)
    out = {}
    for mode in (f16.MATH_STRICT, f16.MATH_FAST):
        prev = f16.lib.f16_set_math_mode(mode)
        for scheme in ("forward", "central"):
            for m in (n, 1, 12):
                fb = f16.F16Batch(x[:, :m], u[:, :m], fi_flag=fi[:m], xcg=xcg[:m])
                A, B, _, _ = fb.linearise(np.ascontiguousarray(x[:, :m]), np.ascontiguousarray(u[:, :m]), scheme=scheme)
                out[mode, scheme, m] = (A, B, fb.last_status.copy(), fb._calc_xdot(np.ascontiguousarray(x[:, :m]), np.ascontiguousarray(u[:, :m])))
        f16.lib.f16_set_math_mode(prev)
    special = np.zeros(n, dtype=bool)
    special[1:9] = True        # the aircraft the fast kernel hands to its reference-order pass
    for scheme in ("forward", "central"):
        for m in (n, 1, 12):
            As, Bs, ss, xd = out[f16.MATH_STRICT, scheme, m]
            Af, Bf, sf, _ = out[f16.MATH_FAST, scheme, m]
            assert np.array_equal(ss, sf), (scheme, m, np.flatnonzero(ss != sf))
            assert np.array_equal(np.isnan(As), np.isnan(Af)) and np.array_equal(np.isnan(Bs), np.isnan(Bf)), (scheme, m)
            sp = special[:m]
            # the redone aircraft carry the strict build's numbers to rounding (same arithmetic, unstaged evaluation order)
            fin = np.isfinite(As[sp])
            d = np.abs(Af[sp][fin] - As[sp][fin])
            assert d.max(initial=0.0) <= 1e-9, (scheme, m, d.max(), np.argwhere(np.abs(np.where(np.isfinite(As), Af - As, 0.0)) > 1e-9)[:5])
            bar = jac_bar(np.where(np.isfinite(xd), xd, 0.0), scheme)
            fa = np.isfinite(As)
            assert (np.abs(Af - As)[fa] <= np.broadcast_to(2 * bar, As.shape)[fa]).all(), (scheme, m)
            fb_ = np.isfinite(Bs)
            assert np.abs(Bf - Bs)[fb_].max(initial=0.0) < 2 * TOL_JAC
    assert out[f16.MATH_FAST, "forward", n][2][1] == 1 << 20 and out[f16.MATH_FAST, "forward", n][2][10] == 1 << 22


def test_linearise_out_of_envelope_column_is_nan(f16, reference_order_linearise):
    g = load_golden("xcg25")
    x = np.repeat(g["x_trim"][:, None], 3, axis=1)
    u = np.repeat(g["u_trim"][:, None], 3, axis=1)
    x[13, 1] = 25.0 - 1e-6     # elevator + eps leaves DH1: that column has no reference answer
    fb = f16.F16Batch(x, u)
    A, B, _, _ = fb.linearise(x, u)
    assert fb.last_status[0] == 0 and fb.last_status[1] == 1 << 20 and fb.last_status[2] == 0
    assert np.isnan(A[1][:, 13]).all() and np.isfinite(A[1][:, 12]).all() and np.isfinite(A[0]).all()


# ---------------------------------------------------------------------------------------------------------
# full BASELINE size through size-independent properties
# ---------------------------------------------------------------------------------------------------------
def test_full_size_batch_properties(f16, oracle, mode):
    """2^20 aircraft (cfg 2 size): a strided sample equals the oracle, the batch equals itself reversed
    (aircraft are independent), and the survivors' checksum is reproducible across two runs"""
    g = load_golden("xcg25")
    n = 1 << 20
    x, u = perturbed_trim(n, g["x_trim"])
    fb = f16.F16Batch(x, u, xcg=0.25)
    fb.step(K=200)
    x1 = fb.x.copy()
    assert (fb.status == 0).mean() > 0.99
    idx = np.arange(0, n, n // 256)
    ref, rst = oracle.step_batch(np.ascontiguousarray(x[:, idx]), np.ascontiguousarray(u[:, idx]), 200, 0.001, 1, 0.25,
                                 None, checker(oracle))
    assert np.array_equal(rst, fb.status[idx])
    assert scaled_err(x1[:, idx], ref) < TOL_TRAJ
    rev = f16.F16Batch(np.ascontiguousarray(x[:, ::-1]), np.ascontiguousarray(u[:, ::-1]), xcg=0.25)
    rev.step(K=200)
    assert np.array_equal(rev.x[:, ::-1], x1)
    fb.reset()
    fb.step(K=200)
    assert np.array_equal(fb.x, x1)


# ---------------------------------------------------------------------------------------------------------
# trim_batch (env.py:198-292): the step before linearise in BASELINE cfg 4
# ---------------------------------------------------------------------------------------------------------
TRIM_SCALE = np.array([1, 1, 1e4, 1, 1, 1, 1e2, 1, 1, 1, 1, 1, 1e3, 1, 1, 1, 1, 1.0])   # natural size of each trim-state entry


def test_trim_matches_reference_golden(f16, mode, golden):
    """F16.trim(10000, 700) of the unmodified reference.  Nelder-Mead amplifies last-bit differences of the objective
    (CUDA's sin/cos/pow vs glibc's) into a different path to the same minimiser: agreement to 1e-6 of each entry's
    natural size -- the reference itself moves by 3e-8 with the tie order of np.argsort (tests/test_oracle.py)."""
    x, opt = f16.trim([10000.0], [700.0], fi=int(golden["fi"]), xcg=float(golden["xcg"]))
    assert opt["success"][0] and opt["status"][0] == 0
    assert np.max(np.abs(x[:, 0] - golden["x_trim"]) / TRIM_SCALE) < 1e-6
    assert 500 < opt["nit"][0] < 5000


@pytest.mark.parametrize("fi", [1, 0])
def test_trim_batch_grid_vs_oracle(f16, oracle, fi):
    """an 8 x 8 altitude x velocity grid (cfg 4 uses 64 x 64 over the same ranges, Nguyen_m/runF16Sim.m:33-39)"""
    hh, vv = np.meshgrid(np.linspace(5000, 40000, 8), np.linspace(300, 900, 8), indexing="ij")
    h, v = hh.ravel(), vv.ravel()
    xr, info, rst = oracle.trim_batch(h, v, fi, 0.35, backend=checker(oracle))
    x, opt = f16.trim(h, v, fi=fi, xcg=0.35)
    assert np.array_equal(opt["status"], rst)
    ok = (rst == 0) & (info[3] != 0)
    assert ok.mean() > 0.9 and np.array_equal(opt["success"][ok], np.ones(ok.sum(), dtype=bool))
    # same minimum: the cost agrees to the objective's own rounding everywhere ...
    assert np.all(np.abs(opt["fun"][ok] - info[0][ok]) <= 1e-6 * info[0][ok] + 1e-12)
    # ... and the same point, to 1e-5 of each entry's natural size where a trim exists (cost ~ 0).  A flight condition
    # that cannot be trimmed (300 ft/s at 35000 ft: cost 0.045, thrust command below its 1000 lb clip, where the objective
    # no longer depends on it) has a flat direction along which two Nelder-Mead runs stop 4e-5 apart.
    err = np.max(np.abs(x - xr) / TRIM_SCALE[:, None], axis=0)
    sharp = ok & (info[0] < 1e-5) & (xr[12] > 1000) & (xr[12] < 19000)
    assert err[ok].max() < 1e-3
    if fi == 1:
        assert sharp.sum() >= 10
    assert not sharp.any() or err[sharp].max() < 1e-5
    # it IS a trim: the weighted derivatives of env.py:258-260, at the clipped point obj_func evaluates (env.py:240-250)
    xc = x[:, ok].copy()
    for i, (lo, hi) in zip((12, 13, 14, 15), ((1000, 19000), (-25, 25), (-21.5, 21.5), (-30, 30))):
        xc[i] = np.clip(xc[i], lo, hi)
    xc[7] = np.clip(xc[7], -20 * np.pi / 180, 90 * np.pi / 180)
    fb = f16.F16Batch(xc, xc[12:16], fi_flag=fi, xcg=0.35)
    xd = fb._calc_xdot(xc, xc[12:16])
    w = np.array([0, 0, 5, 10, 10, 10, 2, 10, 10, 10, 10, 10.0])
    assert np.allclose((w[:, None] * xd[:12] ** 2).sum(axis=0), opt["fun"][ok], rtol=1e-6, atol=1e-14)


def test_trim_then_linearise_full_cfg4_grid(f16):
    """BASELINE cfg 4 end to end on the device: 64 x 64 trims, then central A/B at every trim point"""
    hh, vv = np.meshgrid(np.linspace(5000, 40000, 64), np.linspace(300, 900, 64), indexing="ij")
    x, opt = f16.trim(hh.ravel(), vv.ravel(), fi=1, xcg=0.35)
    ok = opt["success"] & (opt["status"] == 0)
    assert ok.mean() > 0.95
    assert np.all(x[2] == hh.ravel()) and np.all(x[6] == vv.ravel())
    assert np.all(np.abs(x[7, ok]) < np.deg2rad(45)) and np.all((x[12, ok] >= 1000 - 1e-9) | (opt["fun"][ok] > 1e-3))
    fb = f16.F16Batch(x[:, ok], x[12:16, ok], xcg=0.35)
    A, B, _, _ = fb.linearise(x[:, ok], x[12:16, ok], scheme="central")
    assert np.isfinite(A).all() and np.isfinite(B).all() and (fb.last_status == 0).all()
    # actuator block of A is the first-order lags of utils.py:308-330 wherever no rate limit is active
    assert np.allclose(A[:, 13, 13], -20.2) and np.allclose(A[:, 14, 14], -20.2) and np.allclose(A[:, 15, 15], -20.2)


_CFG4_REF = {}


def test_cfg4_full_grid_jacobians_against_the_oracle(f16, oracle, mode):
    """BASELINE cfg 4 at its stated size as a PARITY test (VERDICT r01 weak #4): all 64 x 64 device-computed trim points,
    forward (env.py:294-342, eps 1e-5) and central A/B from linearise_batch -- the strict kernel and, in fast mode, the
    two-aircraft-per-warp kernel on the fast arithmetic -- against the same scheme looped over the reference .so at every
    point (trim points computed once, in strict mode, so that both builds are compared at the same arguments)."""
    if "pts" not in _CFG4_REF:
        prev = f16.lib.f16_set_math_mode(f16.MATH_STRICT)
        hh, vv = np.meshgrid(np.linspace(5000, 40000, 64), np.linspace(300, 900, 64), indexing="ij")
        x, opt = f16.trim(hh.ravel(), vv.ravel(), fi=1, xcg=0.35)
        f16.lib.f16_set_math_mode(prev)
        ok = opt["success"] & (opt["status"] == 0)
        assert ok.sum() >= 4000, int(ok.sum())
        xs, us = np.ascontiguousarray(x[:, ok]), np.ascontiguousarray(x[12:16, ok])
        _CFG4_REF["pts"] = (xs, us)
        for code in (0, 1):
            _CFG4_REF[code] = oracle.linearise_batch(xs.copy(), us.copy(), 1e-5, code, 1, 0.35, checker(oracle))
    xs, us = _CFG4_REF["pts"]
    fb = f16.F16Batch(xs, us, xcg=0.35)
    xd = fb._calc_xdot(xs, us)
    for scheme, code in (("forward", 0), ("central", 1)):
        A, B, _, _ = fb.linearise(xs, us, scheme=scheme)
        rA, rB, rst = _CFG4_REF[code]
        assert np.array_equal(fb.last_status, rst) and not rst.any()
        bar = jac_bar(xd, code)                                                # [N][18][1]
        eA, eB = np.abs(A - rA), np.abs(B - rB)
        assert (eA <= bar).all() and (eB <= bar).all(), (scheme, eA.max(), eB.max(), np.unravel_index(np.argmax(eA - bar), eA.shape))
        over = eA > TOL_JAC
        assert eB.max() < TOL_JAC
        # the allowance is used only by rows whose own value is large: the navigation rows (300 .. 900 ft/s) and, at the few
        # grid corners where Nelder-Mead "trims" with a thrust of -2e5 lb, the V-dot row (|f_6| ~ 300 ft/s^2)
        big = (np.abs(xd).T >= 100.0)[:, :, None]
        assert not (over & ~big).any(), (scheme, np.argwhere(over & ~big)[:4])
        if mode == "strict":
            assert not over[:, 2:, :].any(), (scheme, np.argwhere(over[:, 2:, :])[:4])
        print(f"cfg4 {mode} {scheme}: max |dA| {eA.max():.2e} (rows 0-1: {int(over.sum())} of {over[:, :2].size} entries above 1e-8), "
              f"rows 2..17 max {eA[:, 2:].max():.2e}, max |dB| {eB.max():.2e}")


_BENCH_SAMPLE_CACHE = {}


def _bench_batch_sample(oracle, workload, n, K, n_sample=256):
    """bench.py's own batch for `workload` (same generator, same seed as rank 0) and the oracle's final state of a strided
    sample of it after K Euler steps (cached across the math-mode parametrisation: ~6 s of CPU per workload)."""
    import bench
    from f16_mpc_oop_py_b200.shard import rank_seed
    tag, xcg = ("xcg35", 0.35) if workload == "lqr" else ("xcg25", 0.25)
    x_trim, u_trim, mpc_idx = bench.trim_state(tag)
    x, u = bench.perturbed_trim(n, x_trim, u_trim, seed=rank_seed(0xF16, 0))
    idx = np.arange(0, n, n // n_sample)
    key = (workload, n, K)
    if key not in _BENCH_SAMPLE_CACHE:
        law = None
        if workload == "lqr":
            law = orc_make_lqr(-load_golden(tag)["K_lqr"], mpc_idx, x_trim[mpc_idx], u_trim, rows=[1, 2, 3])
        _BENCH_SAMPLE_CACHE[key] = oracle.step_batch(np.ascontiguousarray(x[:, idx]), np.ascontiguousarray(u[:, idx]), K, 0.001,
                                                     1, xcg, law, checker(oracle))
    return x, u, idx, xcg, x_trim, u_trim, mpc_idx, _BENCH_SAMPLE_CACHE[key]


@pytest.mark.parametrize("workload", ["open", "lqr"])
def test_bench_workload_final_state_sample_against_the_oracle(f16, oracle, mode, workload):
    """VERDICT r01 weak #3: the bench's OWN run -- cfg 2 (2^20 aircraft x 10 000 fused Euler steps, open loop, xcg 0.25) and
    cfg 5's closed loop (u = u0 - K (x - x_trim) with the reference's K_lqr, xcg 0.35, 2^20 of its 8 Mi aircraft per GPU) --
    sampled at 256 aircraft against the reference .so after the full 10 s: <= 1e-9 scaled, status words equal."""
    n, K = 1 << 20, 10000
    x, u, idx, xcg, x_trim, u_trim, mpc_idx, (ref, rst) = _bench_batch_sample(oracle, workload, n, K)
    law = None
    if workload == "lqr":
        law = f16.make_lqr(-load_golden("xcg35")["K_lqr"], mpc_idx, x_trim[mpc_idx], u_trim, rows=[1, 2, 3])
    fb = f16.F16Batch(x, u, xcg=xcg)
    fb.step(K=K, lqr=law)
    st = fb.status[idx]
    # who stopped: the oracle's status word, except an aircraft that crosses a bound within rounding of the last step
    assert int((st != rst).sum()) <= 1, np.flatnonzero(st != rst)
    alive = (st == 0) & (rst == 0)
    assert alive.mean() > (0.95 if workload == "lqr" else 0.9), alive.mean()
    err = scaled_err(fb.x[:, idx][:, alive], ref[:, alive])
    assert err < TOL_TRAJ, err
    assert np.array_equal(fb.steps_done[idx][alive], np.full(int(alive.sum()), K))


def test_trim_fixed_point_exit_is_exact_on_the_cfg4_grid(f16, mode):
    """the 64 x 64 cfg-4 grid at xcg 0.25 (2 % of it never converges): with and without the fixed-point exit of the search the
    same points, costs, iteration and evaluation counts, bit for bit -- and the exit is what makes the grid a 40 ms launch"""
    import time
    hh, vv = np.meshgrid(np.linspace(5000, 40000, 64), np.linspace(300, 900, 64), indexing="ij")
    out = {}
    for on in (1, 0):
        prev = f16.lib.f16_set_trim_fixed_point_exit(on)
        try:
            t0 = time.perf_counter()
            out[on] = f16.trim(hh.ravel(), vv.ravel(), xcg=0.25, maxiter=6000) + (time.perf_counter() - t0,)
        finally:
            f16.lib.f16_set_trim_fixed_point_exit(prev)
    (xa, oa, ta), (xb, ob, tb) = out[1], out[0]
    assert np.array_equal(xa, xb, equal_nan=True)
    for k in ("fun", "nit", "nfev", "success", "status"):
        assert np.array_equal(oa[k], ob[k], equal_nan=True), k
    assert 0 < (~oa["success"]).sum() < 200 and (oa["nit"][~oa["success"]] == 6000).all()
    assert ta < tb


def test_trim_edges(f16):
    x, opt = f16.trim(np.zeros(0), np.zeros(0))
    assert x.shape == (18, 0)
    x, opt = f16.trim([10000.0, 10000.0], [700.0, 700.0], fi=np.array([1, 7], dtype=np.uint8))
    assert opt["status"][0] == 0 and opt["status"][1] == 1 << 22 and np.isnan(x[:, 1]).all()
    x, opt = f16.trim([10000.0], [700.0], maxiter=25)
    assert not opt["success"][0] and opt["nit"][0] == 25


# ---------------------------------------------------------------------------------------------------------
# reduced model, zero-order hold, discrete LQR gain (env.py:46-60,344-358; utils.py:219-245)
# ---------------------------------------------------------------------------------------------------------
def test_reduced_jacobian_is_the_reference_ssr(f16, golden):
    fb = f16.F16Batch(golden["x_trim"], golden["u_trim"], fi_flag=int(golden["fi"]), xcg=float(golden["xcg"]))
    A, B, _, _ = fb.linearise(golden["x_trim"], golden["u_trim"], scheme="forward")
    Ana, Bna = f16.reduce_jacobian(A)
    from oracle import reduce_jacobian
    ra, rb = reduce_jacobian(A)
    assert np.array_equal(Ana, ra) and np.array_equal(Bna, rb)          # the gather itself is exact
    assert np.abs(Ana[0] - golden["na_Ac"]).max() < TOL_JAC and np.abs(Bna[0] - golden["na_Bc"]).max() < TOL_JAC


def test_discretise_matches_cont2discrete(f16, golden):
    from oracle import discretise
    for A, B, Ad_ref, Bd_ref in ((golden["Ac"], golden["Bc"], golden["Ad"], golden["Bd"]),
                                 (golden["na_Ac"], golden["na_Bc"], golden["na_Ad"], golden["na_Bd"])):
        Ad, Bd = f16.discretise(A, B, 0.001)
        scale = max(np.abs(Ad_ref).max(), 1.0)
        assert np.abs(Ad[0] - Ad_ref).max() < 1e-13 * scale and np.abs(Bd[0] - Bd_ref).max() < 1e-13 * scale
    # a stack of random systems, small and large steps (scaling and squaring), against scipy
    r = np.random.default_rng(3)
    A = r.normal(size=(40, 18, 18)) * r.uniform(0.1, 30, size=(40, 1, 1))
    B = r.normal(size=(40, 18, 4))
    for dt in (0.001, 0.05, 0.5):
        Ad, Bd = f16.discretise(A, B, dt)
        for i in range(0, 40, 7):
            ra, rb = discretise(A[i], B[i], dt)
            s = max(np.abs(ra).max(), np.abs(rb).max(), 1.0)
            assert np.abs(Ad[i] - ra).max() < 1e-11 * s and np.abs(Bd[i] - rb).max() < 1e-11 * s


def test_dlqr_matches_reference_gain(f16, golden):
    K, P, info = f16.dlqr(golden["na_Ad"], golden["na_Bd"], np.eye(9), np.eye(3))
    assert info[0, 0] == 0 and 10 < info[0, 1] < 40
    Kref = -golden["K_lqr"]
    assert np.abs(K[0] - Kref).max() < 1e-9 * np.abs(Kref).max()
    from oracle import dlqr
    _, Pref = dlqr(golden["na_Ad"], golden["na_Bd"], np.eye(9), np.eye(3))
    assert np.abs(P[0] - Pref).max() < 1e-9 * np.abs(Pref).max()


def test_lqr_gain_batch_end_to_end(f16, golden):
    """F16._calc_LQR_gain on the device: linearise -> reduce -> cont2discrete -> dlqr, against the reference's own K"""
    fb = f16.F16Batch(golden["x_trim"], golden["u_trim"], fi_flag=int(golden["fi"]), xcg=float(golden["xcg"]))
    K = fb._calc_LQR_gain()
    assert K.shape == (1, 3, 9) and fb.last_status[0] == 0
    # the gain inherits the 1e-10 finite-difference noise of A through a Riccati equation with cond(P) ~ 1e6
    assert np.abs(K[0] - golden["K_lqr"]).max() < 1e-5 * np.abs(golden["K_lqr"]).max()


def test_gain_scheduled_chain_over_a_trim_grid(f16):
    """trim -> linearise -> reduce -> discretise -> dlqr over an 8 x 8 altitude x velocity grid; every closed loop is stable"""
    hh, vv = np.meshgrid(np.linspace(5000, 30000, 8), np.linspace(400, 900, 8), indexing="ij")
    x, opt = f16.trim(hh.ravel(), vv.ravel(), xcg=0.35)
    ok = opt["success"] & (opt["status"] == 0) & (opt["fun"] < 1e-4)
    assert ok.sum() > 40
    fb = f16.F16Batch(x[:, ok], x[12:16, ok], xcg=0.35)
    A, B, _, _ = fb.linearise(fb.x, fb.u, scheme="forward")
    Ana, Bna = f16.reduce_jacobian(A)
    Ad, Bd = f16.discretise(Ana, Bna, 0.001)
    K, P, info = f16.dlqr(Ad, Bd, np.eye(9), np.eye(3))
    assert (info[:, 0] == 0).all()
    for i in range(K.shape[0]):
        rho = np.abs(np.linalg.eigvals(Ad[i] - Bd[i] @ K[i])).max()
        assert rho < 1.0
    Kb = fb._calc_LQR_gain()
    assert np.allclose(Kb, -K, rtol=1e-9, atol=1e-9)


def test_rollout_snapshots_equal_chunked_steps(f16, oracle, mode):
    """step_batch_traj: snapshots every 250 steps of a 1000-step run = the states a user would get by calling step 4 times,
    bit for bit, and the oracle's trajectory within tolerance; closed loop too"""
    g = load_golden("xcg35")
    x, u = perturbed_trim(300, g["x_trim"], seed=17)
    sel = list(g["mpc_x_idx"])
    law = f16.make_lqr(-g["K_lqr"], sel, g["x_trim"][sel], g["u_trim"], rows=[1, 2, 3])
    for lqr in (None, law):
        fb = f16.F16Batch(x, u, xcg=0.35)
        traj = fb.rollout(1000, 250, lqr=lqr)
        fc = f16.F16Batch(x, u, xcg=0.35)
        for s in range(4):
            fc.step(K=250, lqr=lqr)
            assert np.array_equal(traj[s], fc.x)
        assert np.array_equal(fb.x, fc.x) and np.array_equal(fb.status, fc.status)
        olaw = None if lqr is None else orc_make_lqr(-g["K_lqr"], sel, g["x_trim"][sel], g["u_trim"], rows=[1, 2, 3])
        ref, rst = oracle.step_batch(x, u, 500, 0.001, 1, 0.35, olaw, checker(oracle))
        alive = (rst == 0) & (fb.status == 0)
        assert alive.mean() > 0.5 and scaled_err(traj[1][:, alive], ref[:, alive]) < TOL_TRAJ
    # K not a multiple of snap_every: the tail is still integrated
    fb = f16.F16Batch(x, u, xcg=0.35)
    traj = fb.rollout(130, 50)
    fc = f16.F16Batch(x, u, xcg=0.35)
    fc.step(K=130)
    assert traj.shape[0] == 2 and np.array_equal(fb.x, fc.x)


def test_step_on_the_envelope_corners(f16, oracle, mode):
    """one Euler step from states exactly on the edges of every table axis (alpha -20 / 45 deg, beta +-30 deg, dele +-25 deg,
    h 0 / 100000 ft) and within an ulp of interior breakpoints: the cell search of both builds must pick a valid cell"""
    g = load_golden("xcg25")
    d2r = np.pi / 180
    alphas = [-20 * d2r, 45 * d2r, np.nextafter(45 * d2r, 0), 0.0, 5 * d2r, np.nextafter(5 * d2r, 1), np.nextafter(5 * d2r, -1)]
    betas = [-30 * d2r, 30 * d2r, np.nextafter(30 * d2r, 0), -10 * d2r, 10 * d2r, 0.0, np.nextafter(10 * d2r, 1)]
    els = [-25.0, 25.0, -10.0, 10.0, 0.0, np.nextafter(10.0, 0), np.nextafter(-10.0, 0)]
    alts = [0.0, 100000.0, 35000.0, np.nextafter(35000.0, 0), 99999.0]
    cases = []
    for a in alphas:
        for b in betas:
            for e in els:
                x = g["x_trim"].copy()
                x[7], x[8], x[13] = a, b, e
                x[2] = alts[len(cases) % len(alts)]
                cases.append(x)
    x = np.ascontiguousarray(np.array(cases).T)
    u = np.ascontiguousarray(np.tile(g["u_trim"][:, None], (1, x.shape[1])))
    ref, rst = oracle.step_batch(x, u, 1, 0.001, 1, 0.25, None, checker(oracle))
    fb = f16.F16Batch(x, u, xcg=0.25)
    fb.step(K=1)
    assert np.array_equal(fb.status, rst)
    ok = rst == 0
    assert ok.sum() > 200
    assert np.all(np.abs(fb.x[:, ok] - ref[:, ok]) <= 1e-13 * np.maximum(np.abs(ref[:, ok]), 1.0))
    assert np.array_equal(fb.x[:, ~ok], x[:, ~ok])      # stopped aircraft keep their state

def _dt1_derivative_error(f16, oracle, x, u, xcg, fi=1):
    """One Euler step with dt = 1.0 through step_batch, so that x1 - x0 IS the derivative the step kernel computed (a
    derivative error is not scaled down by dt = 1e-3): |x1 - fl(x0 + xdot_ref)| in units of max(|xdot_ref|, rms of that
    derivative over the batch), after allowing the one rounding of the sum (1 ulp of x1)."""
    ref, rst = oracle.calc_xdot_batch(x, u, fi, xcg, checker(oracle))
    fb = f16.F16Batch(x, u, fi_flag=fi, xcg=xcg, dt=1.0)
    fb.step(K=1)
    assert np.array_equal(fb.status, np.zeros_like(fb.status)) and not rst.any()
    assert (fb.steps_done == 1).all() and np.isfinite(fb.x).all()
    want = x + ref
    scale = np.maximum(np.abs(ref), np.sqrt(np.mean(ref * ref, axis=1, keepdims=True)))
    scale = np.where(scale == 0, 1.0, scale)
    excess = np.maximum(np.abs(fb.x - want) - np.spacing(np.abs(want)), 0.0)
    return excess / scale


@pytest.mark.parametrize("xcg", [0.25, 0.35])
def test_step_kernel_derivative_in_the_breakpoint_bands(f16, oracle, mode, xcg):
    """VERDICT r01 #1/#2: the derivative of the STEP kernels (in fast mode: f16_fast.cuh on the device, with the device's own
    rcp / sincos code) at alpha, beta, elevator on every interior breakpoint, +-1 ulp and +-{1e-12 .. 1e-6} of a cell width,
    <= 1e-12 scaled against the reference .so.  dt = 1 makes x1 - x0 the derivative."""
    from _inputs import breakpoint_band_states
    x = breakpoint_band_states(X_TRIM_XCG25)
    u = np.ascontiguousarray(np.tile(X_TRIM_XCG25[12:16][:, None], (1, x.shape[1])))
    err = _dt1_derivative_error(f16, oracle, x, u, xcg)
    w = np.unravel_index(np.argmax(err), err.shape)
    assert err.max() < TOL_DERIV, (err.max(), w, x[[7, 8, 13], w[1]] * [180 / np.pi, 180 / np.pi, 1])


@pytest.mark.parametrize("fi", [1, 0])
def test_step_kernel_derivative_over_the_envelope(f16, oracle, mode, fi):
    """the same dt = 1 derivative check of the step kernels on 20 000 random in-envelope states and on perturbed-trim
    states (VERDICT r01 weak #2: the device-side 1e-12 check of the arithmetic that carries the headline number)"""
    n = 20000
    xu = random_envelope_xu(n, seed=23, hifi=bool(fi))
    r = np.random.default_rng(6)
    x = np.vstack([xu, r.uniform(-30, 30, (1, n))])
    x[2] = r.uniform(0, 60000, n)
    u = np.stack([r.uniform(500, 20000, n), r.uniform(-30, 30, n), r.uniform(-25, 25, n), r.uniform(-35, 35, n)])
    err = _dt1_derivative_error(f16, oracle, np.ascontiguousarray(x), np.ascontiguousarray(u), 0.25, fi)
    assert err.max() < TOL_DERIV, (err.max(), np.unravel_index(np.argmax(err), err.shape))
    xp, up = perturbed_trim(n, X_TRIM_XCG25, seed=12)
    err = _dt1_derivative_error(f16, oracle, xp, up, 0.35, fi)
    assert err.max() < TOL_DERIV, (err.max(), np.unravel_index(np.argmax(err), err.shape))


@pytest.mark.parametrize("xcg", [0.25, 0.35])
def test_calc_xdot_in_the_breakpoint_bands(f16, oracle, mode, xcg):
    """calc_xdot_batch (the one-shot kernels) on the same band states, both builds"""
    from _inputs import breakpoint_band_states
    x = breakpoint_band_states(X_TRIM_XCG25)
    u = np.ascontiguousarray(np.tile(X_TRIM_XCG25[12:16][:, None], (1, x.shape[1])))
    ref, rst = oracle.calc_xdot_batch(x, u, 1, xcg, checker(oracle))
    fb = f16.F16Batch(x, u, xcg=xcg)
    out = fb._calc_xdot(x, u)
    assert not rst.any() and not fb.last_status.any()
    assert scaled_err(out, ref) < TOL_DERIV


def test_integer_pipe_comparisons_on_their_thresholds(f16, oracle, mode):
    """The comparisons that f16_fast.cuh asks on the integer pipe -- airspeed floor (nlplant.c:104), tropopause (nlplant.c:475), the
    five actuator rate limits (utils.py:299-330) -- ON, one ulp either side of and well either side of their thresholds: the
    derivative of the step kernel (dt = 1) and of the one-shot kernel against the reference .so, both builds."""
    from _inputs import comparison_threshold_cases
    x, u = comparison_threshold_cases(X_TRIM_XCG25, oracle.atmos)
    ref, rst = oracle.calc_xdot_batch(x, u, 1, 0.25, checker(oracle))
    assert not rst.any()
    for row, lim in ((12, 10000.0), (13, 60.0), (14, 80.0), (15, 120.0), (16, 25.0)):
        assert (np.abs(ref[row]) == lim).any() and (np.abs(ref[row]) < lim).any(), row
    fb = f16.F16Batch(x, u, xcg=0.25)
    out = fb._calc_xdot(x, u)
    assert not fb.last_status.any()
    assert scaled_err(out, ref) < TOL_DERIV
    # the step kernel: an airspeed of 0 is ON a state bound (exact path of the screen) and steps like any other
    err = _dt1_derivative_error(f16, oracle, x, u, 0.25)
    assert err.max() < TOL_DERIV, (err.max(), np.unravel_index(np.argmax(err), err.shape))
    # and in a batch large enough for the TMA-tiled kernels (the same states, repeated)
    reps = 4096 // x.shape[1] + 1
    xb, ub = np.ascontiguousarray(np.tile(x, (1, reps))), np.ascontiguousarray(np.tile(u, (1, reps)))
    fb = f16.F16Batch(xb, ub, xcg=0.25)
    outb = fb._calc_xdot(xb, ub)
    assert scaled_err(outb, np.tile(ref, (1, reps))) < TOL_DERIV


# ---------------------------------------------------------------------------------------------------------
# end-of-run statistics reduced on the device (f16_stats.cu; SURVEY 8e / 8f rank 4)
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 31, 257, 100003])
def test_state_summary_matches_numpy(f16, n):
    from f16_mpc_oop_py_b200 import shard
    r = np.random.default_rng(n)
    g = load_golden("xcg25")
    x, _ = perturbed_trim(n, g["x_trim"], seed=n, frac=0.05)
    x[0] = r.uniform(-1e4, 1e4, n)                      # a plane whose mean is far from its spread
    x[2] = 1e4 + 1e-3 * r.standard_normal(n)            # ... and one where sum-of-squares formulas cancel
    st = (r.uniform(size=n) < 0.2).astype(np.int32) * 4
    for status in (None, st):
        row = f16.state_summary(x, status)
        ref = shard.summarise(x, np.zeros(n, dtype=np.int32) if status is None else status)
        assert row[0] == n and row[1] == ref[1]
        if ref[1] == 0:
            assert np.all(np.isposinf(row[2:20])) and np.all(np.isneginf(row[20:38])) and not row[38:].any()
            continue
        assert np.array_equal(row[2:38], ref[2:38])                                   # min, max: exact
        # mean: 1e-13 of the size of the data (|mean| or the rms of the plane, as for every other parity metric here -- the
        # plane of +-1e4 uniform values has a mean of ~30 and no digits to spare below 1e-12 in EITHER summation order)
        xa = x if status is None else x[:, status == 0]
        scale = np.maximum(np.abs(ref[38:56]), np.sqrt((xa * xa).mean(axis=1)))
        assert np.all(np.abs(row[38:56] - ref[38:56]) <= 1e-13 * scale + 1e-300)
        assert np.allclose(row[56:74], ref[56:74], rtol=1e-10, atol=1e-18)           # M2 (one shifted pass vs numpy's two)
    assert np.array_equal(f16.state_summary(x, st), f16.state_summary(x, st))        # fixed reduction tree


@pytest.mark.gpu
def test_state_summary_edges_and_batch_method(f16):
    row = f16.state_summary(np.zeros((18, 0)))
    assert row[0] == 0 and row[1] == 0 and np.all(np.isposinf(row[2:20])) and not row[38:].any()
    g = load_golden("xcg25")
    x, u = perturbed_trim(2000, g["x_trim"], seed=3, frac=0.05)
    fb = f16.F16Batch(x, u, xcg=0.25)
    fb.step(K=50)
    from f16_mpc_oop_py_b200 import shard
    ref = shard.summarise(fb.x, fb.status)
    row = fb.summary()
    assert row[1] == ref[1] and np.array_equal(row[2:38], ref[2:38]) and np.allclose(row[38:56], ref[38:56], rtol=1e-13)
    merged = shard.merge_summaries([row])
    assert merged["alive"] == int(ref[1])

@pytest.mark.gpu
def test_rollout_stats_equals_chunked_steps_and_summaries(f16, mode):
    """step_batch_stats: statistics every M steps without trajectories = step(M) + summary(), repeated, bit for bit"""
    g = load_golden("xcg35")
    n, K, M = 3000, 240, 40
    x, u = perturbed_trim(n, g["x_trim"], seed=12, frac=0.05)
    x[7, :40] = np.deg2rad(44.9)                      # near the edge of the tables
    x[7, 40:60] = np.deg2rad(46.0)                    # outside them: frozen from the first step, not in the statistics
    a = f16.F16Batch(x, u, xcg=0.35)
    rows = a.rollout_stats(K, M)
    assert rows.shape == (K // M, 74)
    b = f16.F16Batch(x, u, xcg=0.35)
    for i in range(K // M):
        b.step(K=M)
        assert np.array_equal(rows[i], b.summary(), equal_nan=True), i
    assert np.array_equal(a.x, b.x, equal_nan=True) and np.array_equal(a.status, b.status)
    assert rows[0][0] == n and rows[-1][1] == (b.status == 0).sum() and 0 < rows[-1][1] < n
    assert np.all(np.diff(rows[:, 1]) <= 0)           # survivors never come back

@pytest.mark.gpu
def test_step_beyond_2_to_31_elements(f16):
    """maximum sizes: 2^27 + 5 aircraft -- plane offsets pass 2^31 elements (17 x 2^27 = 2.3e9), 19 GB of state built on the
    device by tiling a 2^20-aircraft block; the tiles must come out of the step bit-identical to that block run alone"""
    import ctypes
    L = f16.lib
    g = load_golden("xcg25")
    nb = 1 << 20
    reps = 128
    n = nb * reps + 5
    xb, ub = perturbed_trim(nb + 5, g["x_trim"], seed=99, frac=0.05)
    small = f16.F16Batch(xb, ub, xcg=0.25)
    small.step(K=7)
    d_x, d_u, d_st = L.f16_dev_alloc(18 * n * 8), L.f16_dev_alloc(4 * n * 8), L.f16_dev_alloc(4 * n)
    if not (d_x and d_u and d_st):
        pytest.skip("not enough device memory for the 19 GB batch")
    try:
        for arr, d, planes in ((xb, d_x, 18), (ub, d_u, 4)):
            for i in range(planes):
                base = d + (i * n) * 8
                assert L.f16_memcpy_h2d(base, arr[i, :nb].ctypes.data, nb * 8) == 0
                filled = nb
                while filled < nb * reps:                      # doubling device-to-device copies
                    c = min(filled, nb * reps - filled)
                    assert L.f16_memcpy_d2d(base + filled * 8, base, c * 8) == 0
                    filled += c
                tail = np.ascontiguousarray(arr[i, nb:nb + 5])
                assert L.f16_memcpy_h2d(base + nb * reps * 8, tail.ctypes.data, 5 * 8) == 0
        assert L.step_batch_dev(d_x, n, d_u, n, n, 7, 0.001, None, None, 1, None, 0.25, d_st, None) == 0
        row = f16.state_summary_dev(d_x, n, n, d_st)
        assert row[0] == n and row[1] == reps * int((small.status[:nb] == 0).sum()) + int((small.status[nb:] == 0).sum())
        out = np.empty(nb)
        for i in (0, 7, 17):                                    # first, a middle and the last plane (offset 17 n > 2^31)
            for tile in (0, 77, reps - 1):
                assert L.f16_memcpy_d2h(out.ctypes.data, d_x + (i * n + tile * nb) * 8, nb * 8) == 0
                assert np.array_equal(out, small.x[i, :nb], equal_nan=True), (i, tile)
            t5 = np.empty(5)
            assert L.f16_memcpy_d2h(t5.ctypes.data, d_x + (i * n + reps * nb) * 8, 5 * 8) == 0
            assert np.array_equal(t5, small.x[i, nb:], equal_nan=True)
    finally:
        for p in (d_x, d_u, d_st):
            L.f16_dev_free(p)

@pytest.mark.gpu
def test_division_helpers_have_the_bits_of_the_device_division(f16):
    """F16_DIV (the division sequence without its range test and slow-path branch) and div_by (rounded reciprocal + one
    residual correction) against a / b ON THE DEVICE: ordinary operands over 60 decades, the model's own divisors (vt,
    cos(theta), U^2 + W^2, ps), zero numerators, and numerators whose quotient sits on a rounding midpoint"""
    import random
    from fractions import Fraction  # noqa: F401
    sys_path_tests = os.path.dirname(os.path.abspath(__file__))
    import importlib.util
    spec = importlib.util.spec_from_file_location("ted", os.path.join(sys_path_tests, "test_exact_division.py"))
    ted = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ted)
    r = np.random.default_rng(17)
    rnd = random.Random(17)
    n = 2_000_000
    a = r.uniform(-1, 1, n) * 10.0 ** r.integers(-30, 30, n)
    b = r.uniform(0.5, 1, n) * 10.0 ** r.integers(-30, 30, n) * r.choice([-1.0, 1.0], n)
    a[:1000] = 0.0
    b[1000:200000] = r.uniform(0.01, 900, 199000)                    # vt
    b[200000:400000] = np.cos(r.uniform(-1.57, 1.57, 200000))        # cos(theta)
    b[400000:600000] = r.uniform(1e-4, 1e6, 200000)                  # U^2 + W^2
    k = 600000
    for y in (700.0, 0.9999, 11.32, 2116.2, 3.7e5) + tuple(r.uniform(0.01, 1e6, 40)):
        hard = np.array(ted.hard_numerators(float(y), 2000, rnd))
        a[k:k + hard.size] = hard
        b[k:k + hard.size] = y
        k += hard.size
    out = np.empty((3, n))
    assert f16.lib.f16_div_probe(a.ctypes.data, b.ctypes.data, n, out.ctypes.data) == 0
    with np.errstate(all="ignore"):
        host = a / b
    assert np.array_equal(out[2].view(np.uint64), host.view(np.uint64))          # the device divides as IEEE 754 says
    assert np.array_equal(out[0], out[2])                                        # values (a zero keeps its value, not its sign)
    nz = a != 0
    assert np.array_equal(out[0][nz].view(np.uint64), out[2][nz].view(np.uint64))
    assert np.array_equal(out[1].view(np.uint64), out[2].view(np.uint64))

