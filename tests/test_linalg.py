"""The small dense algebra of csrc/f16_linalg.cu -- zero-order hold, discrete LQR by structured doubling, the reduced-model
gather -- against plain high-precision references: mpmath's expm at 40 digits, scipy's cont2discrete and
solve_discrete_are, and the Riccati residual from its definition.

Every case runs on two backends.  "host" is csrc/f16_linalg.cuh compiled for the CPU (tests/hostemu, no FMA contraction) and
runs without a GPU; "device" is libf16_b200.so (linalg.o, FMA-contracted) on the B200.  The two agree to rounding, not bit
for bit, so both face the same bars.  The bars are set from the worst errors measured on the host build (quoted in each
docstring), with at most 10x margin."""
import ctypes
import functools
import os
import subprocess

import numpy as np
import pytest
import scipy.linalg
from scipy.signal import cont2discrete

from conftest import REPO, load_golden
from oracle import NA_COLS, NA_ROWS, NA_UCOLS

SHAPES = [(n, m) for n in range(1, 19) for m in range(1, 23 - n)]  # every (n, m) the entry points accept: 225
MAX_DOUBLINGS, TOL = 64, 1e-15  # the library's dlqr settings (f16_api.cu)
F16_OK, F16_ERR_ARG = 0, -3
ST_OK, ST_NOT_CONVERGED, ST_R_SINGULAR, ST_NONFINITE, ST_NOT_STABILISING, ST_NOT_A_SOLUTION = 0, 1, -1, -3, -5, -6


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


@functools.lru_cache(maxsize=None)
def _hostemu():
    d = os.path.join(REPO, "tests", "hostemu")
    subprocess.check_call(["make", "-s", "-C", d])
    E = ctypes.CDLL(os.path.join(d, "libf16_hostemu.so"))
    vp, i, ll, dbl = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_double
    E.emu_zoh.argtypes = [vp, vp, i, i, ll, dbl, vp, vp]
    E.emu_dlqr.argtypes = [vp, vp, vp, vp, i, i, ll, i, dbl, vp, vp, vp]
    E.emu_reduce_jacobian.argtypes = [vp, ll, vp, vp]
    for f in (E.emu_zoh, E.emu_dlqr, E.emu_reduce_jacobian):
        f.restype = None
    return E


def _stack(A, B):
    A, B = np.ascontiguousarray(A, dtype=np.float64), np.ascontiguousarray(B, dtype=np.float64)
    return A.reshape((-1,) + A.shape[-2:]), B.reshape((-1,) + B.shape[-2:])


class HostLinalg:
    """f16_linalg.cuh on the CPU, same call shapes as f16.discretise / f16.dlqr / f16.reduce_jacobian"""

    def __init__(self):
        self.E = _hostemu()

    def zoh(self, A, B, dt):
        A, B = _stack(A, B)
        n, m = A.shape[1], B.shape[2]
        Ad, Bd = np.empty_like(A), np.empty_like(B)
        self.E.emu_zoh(_p(A), _p(B), n, m, A.shape[0], float(dt), _p(Ad), _p(Bd))
        return Ad, Bd

    def dlqr(self, A, B, Q, R, max_doublings=MAX_DOUBLINGS, tol=TOL):
        A, B = _stack(A, B)
        N, n, m = A.shape[0], A.shape[1], B.shape[2]
        Q = np.ascontiguousarray(Q, dtype=np.float64).reshape(n, n)
        R = np.ascontiguousarray(R, dtype=np.float64).reshape(m, m)
        K, P = np.empty((N, m, n)), np.empty((N, n, n))
        info = np.zeros((N, 2), dtype=np.int32)
        self.E.emu_dlqr(_p(A), _p(B), _p(Q), _p(R), n, m, N, max_doublings, tol, _p(K), _p(P), _p(info))
        return K, P, info

    def reduce_jacobian(self, A):
        A = np.ascontiguousarray(A, dtype=np.float64).reshape(-1, 18, 18)
        Ana, Bna = np.empty((A.shape[0], 9, 9)), np.empty((A.shape[0], 9, 3))
        self.E.emu_reduce_jacobian(_p(A), A.shape[0], _p(Ana), _p(Bna))
        return Ana, Bna


class DeviceLinalg:
    """the library's host-buffer entry points"""

    def __init__(self, f16):
        self.zoh, self.dlqr, self.reduce_jacobian = f16.discretise, f16.dlqr, f16.reduce_jacobian


@pytest.fixture(params=["host", pytest.param("device", marks=pytest.mark.gpu)])
def backend(request):
    return HostLinalg() if request.param == "host" else DeviceLinalg(request.getfixturevalue("f16"))


def _rel(x, ref):
    return float(np.abs(x - ref).max() / max(np.abs(ref).max(), 1.0))


# ---------------------------------------------------------------------------------------------------------------------
# zero-order hold
# ---------------------------------------------------------------------------------------------------------------------
def test_zoh_every_shape_matches_cont2discrete(backend):
    """All 225 accepted (n, m), A ~ 3 N(0, 1), dt in {1e-3, 0.1, 1}: [Ad Bd] within 3e-12 of scipy's cont2discrete,
    relative to the largest entry (or 1).  Measured worst on the host build: 4.8e-13 (n = 4, m = 18, dt = 1); scipy's own
    Pade approximant contributes to it."""
    r = np.random.default_rng(11)
    worst = (0.0, None)
    for n, m in SHAPES:
        A, B = 3 * r.standard_normal((n, n)), r.standard_normal((n, m))
        for dt in (1e-3, 0.1, 1.0):
            Ad, Bd = backend.zoh(A, B, dt)
            ra, rb = cont2discrete((A, B, np.eye(n), np.zeros((n, m))), dt)[:2]
            e = _rel(np.hstack([Ad[0], Bd[0]]), np.hstack([ra, rb]))
            worst = max(worst, (e, (n, m, dt)), key=lambda w: w[0])
    assert worst[0] < 3e-12, worst


def _zoh_cases():
    """(name, A, B, dt, bar): random blocks with ||M||_1 = ||[A B; 0 0] dt||_1 from 1e-4 to 1e3 (0 to 12 squarings), a stiff
    diagonal (||M||_1 = 1e3), non-normal Jordan-like blocks (the stiff 2x2 one reaches ||M||_1 = 5000, 14 squarings), norms
    on and next to the power-of-two scaling boundaries.  The bar is on the error relative to the largest entry (or 1),
    about 5x the worst measured on the host build (in the comments)."""
    r = np.random.default_rng(5)
    cases = []
    for target, n, m in [(1e-4, 3, 1), (1e-3, 6, 2), (1e-2, 4, 4), (0.1, 9, 3), (0.3, 5, 2), (0.49, 8, 3), (0.9, 7, 1),
                         (1.7, 9, 3), (3.9, 6, 2), (8.0, 10, 2), (30.0, 9, 3), (100.0, 5, 3), (300.0, 8, 4), (1000.0, 6, 2),
                         (2.5, 18, 4), (60.0, 18, 4)]:
        # the skew-symmetric part sets the norm; exp stays bounded because the eigenvalues' real parts are O(1) or less
        X = r.standard_normal((n, n))
        A = X - X.T + 0.3 * r.standard_normal((n, n)) - np.eye(n)
        B = r.standard_normal((n, m))
        dt = target / np.abs(np.vstack([np.hstack([A, B]), np.zeros((m, n + m))])).sum(axis=0).max()
        cases.append((f"norm{target:g}_{n}x{m}", A, B, dt, 3e-14))  # measured worst 4.9e-15 (||M||_1 = 300)
    cases.append(("stiff_diagonal", np.diag([-1e4, -1e2, -1.0, -1e-2]), np.ones((4, 1)), 0.1, 2e-13))  # 3.8e-14
    J = -np.eye(3) + np.diag([1e3, 1e3], 1)
    cases.append(("jordan_like_3x3", J, np.array([[0.0], [0.0], [1.0]]), 1.0, 1e-12))  # 1.4e-13
    cases.append(("stiff_nonnormal_2x2", np.array([[-1000.0, 1e4], [0.0, -1.0]]), np.ones((2, 1)), 0.5, 3e-12))  # 6.1e-13
    # dyadic entries: column sums exact, ||M||_1 = 0.5 exactly (no scaling), then 8 exactly and the double just below it
    Ab, Bb = np.array([[-0.25, 0.25], [0.125, -0.25]]), np.array([[0.125], [0.25]])
    cases.append(("norm_exactly_0.5", Ab, Bb, 1.0, 3e-15))  # 0
    cases.append(("norm_above_0.5", Ab, Bb, np.nextafter(1.0, 2.0), 3e-15))  # 1.1e-16
    cases.append(("norm_exactly_8", Ab, Bb, 16.0, 3e-15))  # 4.5e-16
    cases.append(("norm_below_8", Ab, Bb, np.nextafter(16.0, 0.0), 3e-15))  # 1.1e-16
    return cases


ZOH_CASES = _zoh_cases()


@functools.lru_cache(maxsize=None)
def _mp_zoh(k):
    """[Ad Bd] of case k by mpmath.expm at 40 digits, of exactly the double-precision block the kernels exponentiate"""
    import mpmath
    _, A, B, dt, _ = ZOH_CASES[k]
    n, m = B.shape
    M = np.zeros((n + m, n + m))
    M[:n, :n], M[:n, n:] = A * dt, B * dt
    with mpmath.workdps(40):
        E = mpmath.expm(mpmath.matrix(M.tolist()))
        return np.array([[float(E[i, j]) for j in range(n + m)] for i in range(n)])


def test_zoh_matches_mpmath_expm(backend):
    """23 cases against mpmath.expm at 40 digits, each within its bar (_zoh_cases)"""
    fails = []
    for k, (name, A, B, dt, bar) in enumerate(ZOH_CASES):
        Ad, Bd = backend.zoh(A, B, dt)
        e = _rel(np.hstack([Ad[0], Bd[0]]), _mp_zoh(k))
        if not e < bar:
            fails.append((name, e, bar))
    assert not fails, fails


def test_zoh_dt_zero_is_exactly_identity(backend):
    r = np.random.default_rng(2)
    for n, m in ((1, 1), (9, 3), (18, 4), (1, 21)):
        Ad, Bd = backend.zoh(r.standard_normal((2, n, n)), r.standard_normal((2, n, m)), 0.0)
        assert np.array_equal(Ad, np.broadcast_to(np.eye(n), Ad.shape)) and np.array_equal(Bd, np.zeros_like(Bd))


# ---------------------------------------------------------------------------------------------------------------------
# discrete LQR
# ---------------------------------------------------------------------------------------------------------------------
def _weights(r, n, m):
    """non-diagonal symmetric Q >= 0.1 I, R >= 0.5 I (exactly symmetric)"""
    X, Y = r.standard_normal((n, n)), r.standard_normal((m, m))
    Q, R = X @ X.T / n + 0.1 * np.eye(n), Y @ Y.T / m + 0.5 * np.eye(m)
    return (Q + Q.T) / 2, (R + R.T) / 2


def _systems(r, n, m, rho, count):
    """`count` random (A, B) with spectral radius rho(A) = rho"""
    A = r.standard_normal((count, n, n))
    A *= rho / np.abs(np.linalg.eigvals(A)).max(axis=1)[:, None, None]
    return A, r.standard_normal((count, n, m))


def dare_residual(A, B, Q, R, P):
    """||A'PA - P - A'PB (R + B'PB)^-1 B'PA + Q||_F / (||Q||_F + ||A||_2^2 ||P||_F)"""
    S = R + B.T @ P @ B
    res = A.T @ P @ A - P - A.T @ P @ B @ np.linalg.solve(S, B.T @ P @ A) + Q
    return np.linalg.norm(res) / (np.linalg.norm(Q) + np.linalg.norm(A, 2) ** 2 * np.linalg.norm(P))


def check_solution(A, B, Q, R, K, P, info, bar_res=1e-13):
    """what every system with info == 0 must satisfy: P exactly symmetric (the kernel symmetrises), PSD to rounding, the
    Riccati residual at rounding level, A - BK stable"""
    assert info[0] == ST_OK, info
    assert np.array_equal(P, P.T)
    assert np.linalg.eigvalsh(P).min() >= -1e-13 * np.abs(P).max()
    res = dare_residual(A, B, Q, R, P)
    assert res < bar_res, res
    assert np.abs(np.linalg.eigvals(A - B @ K)).max() < 1.0
    return res


def test_dlqr_every_shape(backend):
    """All 225 (n, m), m up to 22 - n (n = 1, m = 21 included), non-diagonal Q and R, three systems per class, on every
    one info 0 and check_solution.  Measured worst on the host build, and the bars:
      well-conditioned, rho(A) = 0.9: P and K within 2.0e-14 of scipy relative to their largest entry (bar 1e-13),
        normalised residual 2.6e-15 (bar 2e-14);
      open-loop unstable, rho(A) = 1.3: normalised residual 4.0e-13 (bar 3e-12), at n = 16, m = 1, where one input holds
        16 modes and |P| is large.  P is not compared with scipy here: the residual is the conditioning-free bar."""
    r = np.random.default_rng(7)
    for n, m in SHAPES:
        Q, R = _weights(r, n, m)
        for rho, bar_res in ((0.9, 2e-14), (1.3, 3e-12)):
            A, B = _systems(r, n, m, rho, 3)
            K, P, info = backend.dlqr(A, B, Q, R)
            for i in range(3):
                check_solution(A[i], B[i], Q, R, K[i], P[i], info[i], bar_res)
                if rho < 1:
                    Pr = scipy.linalg.solve_discrete_are(A[i], B[i], Q, R)
                    Kr = np.linalg.solve(B[i].T @ Pr @ B[i] + R, B[i].T @ Pr @ A[i])
                    e = max(_rel(P[i], Pr), _rel(K[i], Kr))
                    assert e < 1e-13, (n, m, i, e)


def test_dlqr_f16_reduced_model(backend, golden):
    """the golden reduced F-16 model at dt = 1 ms, Q = I, R = I (the gain of cfg 4/5): P within 1.6e-11 of scipy
    (bar 1e-10), normalised residual 2.4e-17 (bar 1e-15)"""
    A, B = golden["na_Ad"], golden["na_Bd"]
    K, P, info = backend.dlqr(A, B, np.eye(9), np.eye(3))
    check_solution(A, B, np.eye(9), np.eye(3), K[0], P[0], info[0], 1e-15)
    assert _rel(P[0], scipy.linalg.solve_discrete_are(A, B, np.eye(9), np.eye(3))) < 1e-10


def test_dlqr_f16_model_under_single_state_weights(backend):
    """xcg 0.35 golden reduced model under each of the nine single-state weights Q = e_k e_k'.  Its eigenvalues near 1
    (1 + 3e-9, 1 + 4.8e-5) are weakly controllable and weakly weighted: doubling takes up to 37 steps and the closed loop
    keeps an eigenvalue within 2.5e-10 of the unit circle.  Every one must converge to the stabilising solution (info 0,
    never -5 or -6).  The residual is only as good as the conditioning allows here: measured worst 2.5e-7 (bar 2e-6).
    (The kernel's own residual test sits at 1e-5 of the terms' size; measured here at most 1.1e-7 -- not checked by this
    test, the kernel does not expose it.)"""
    g = load_golden("xcg35")
    A, B = g["na_Ad"], g["na_Bd"]
    for k in range(9):
        Q = np.diag(np.eye(9)[k])
        K, P, info = backend.dlqr(A, B, Q, np.eye(3))
        check_solution(A, B, Q, np.eye(3), K[0], P[0], info[0], 2e-6)


def test_dlqr_flags_the_marginal_mode_it_leaves_unstable(backend):
    """xcg 0.25 golden reduced model: its eigenvalue 1 + 2e-10 is weighted by none of Q = e_k e_k', k in {0, 2, 3, 4, 6},
    so the doubling converges to the P that leaves it at 1 + 2e-10 (scipy's moves it to 1 - 2e-10).  That is -5 with K
    NaN; P is still written, and its closed loop is indeed unstable.  The other four weights are stabilising: info 0."""
    g = load_golden("xcg25")
    A, B = g["na_Ad"], g["na_Bd"]
    for k in range(9):
        Q = np.diag(np.eye(9)[k])
        K, P, info = backend.dlqr(A, B, Q, np.eye(3))
        if k in (0, 2, 3, 4, 6):
            assert info[0, 0] == ST_NOT_STABILISING and np.isnan(K).all(), (k, info)
            Kp = np.linalg.solve(B.T @ P[0] @ B + np.eye(3), B.T @ P[0] @ A)
            assert np.abs(np.linalg.eigvals(A - B @ Kp)).max() > 1.0
        else:
            check_solution(A, B, Q, np.eye(3), K[0], P[0], info[0], 2e-6)


def test_dlqr_flags_a_doubling_that_broke_down(backend):
    """lofi xcg 0.25 golden reduced model under Q = e_5 e_5' and e_2 e_2': an undetectable mode (1.014) grows A_k and G past
    1e90, I + GH loses all its digits, and the doubling "converges" to an H that is not a solution (normalised residual
    1.5e-3 and 2.9e-3, closed loop unstable).  It must not be reported 0: the kernel's residual test gives -6 (measured
    5.6e-4 and 1.2e-3 of the terms' size, threshold 1e-5).  Every weight whose info is 0 is a checked solution."""
    g = load_golden("lofi_xcg25")
    A, B = g["na_Ad"], g["na_Bd"]
    for k in range(9):
        Q = np.diag(np.eye(9)[k])
        K, P, info = backend.dlqr(A, B, Q, np.eye(3))
        if k in (2, 5):
            assert info[0, 0] == ST_NOT_A_SOLUTION and np.isnan(K).all(), (k, info)
        elif info[0, 0] == ST_OK:
            check_solution(A, B, Q, np.eye(3), K[0], P[0], info[0], 2e-6)
        else:
            assert info[0, 0] < 0 and np.isnan(K).all(), (k, info)


def test_dlqr_slow_unweighted_stable_modes_are_not_flagged(backend):
    """H meets its tolerance while the doubled matrix A_k is still large when a slow stable mode carries no weight (it
    then carries no P).  Those solutions stabilise A - BK and must come back as info 0 with the exact gain: Q = 0 with a
    stable A gives P = 0, K = 0; A = diag(0.1, 0.99) or diag(0.5, 0.9999) under Q = diag(1, 0) keeps the slow mode at
    0.99 / 0.9999 in the closed loop"""
    for A in (np.array([[0.9]]), np.diag([0.9, 0.5])):
        n = A.shape[0]
        K, P, info = backend.dlqr(A, np.eye(n), np.zeros((n, n)), np.eye(n))
        assert info[0, 0] == ST_OK, info
        assert np.array_equal(K[0], np.zeros((n, n))) and np.array_equal(P[0], np.zeros((n, n)))
    for a, b in ((0.1, 0.99), (0.5, 0.9999)):
        A, Q = np.diag([a, b]), np.diag([1.0, 0.0])
        K, P, info = backend.dlqr(A, np.eye(2), Q, np.eye(2))
        check_solution(A, np.eye(2), Q, np.eye(2), K[0], P[0], info[0])
        Pr = scipy.linalg.solve_discrete_are(A, np.eye(2), Q, np.eye(2))
        assert _rel(P[0], Pr) < 1e-13 and abs(np.abs(np.linalg.eigvals(A - K[0])).max() - b) < 1e-15


def test_dlqr_undetectable_unstable_mode_is_flagged(backend):
    """A = diag(1.5, 0.5), B = I, Q = diag(0, 1): the unstable mode carries no weight, so doubling from H0 = Q converges
    to P = diag(0, 1.1328), whose K leaves eigenvalue 1.5 in A - BK (scipy's stabilising P is diag(1.25, 1.1328)).  It
    must be flagged -5 with K NaN; P is still written.  Same for an undetectable eigenvalue of 1.0001."""
    for a in (1.5, 1.0001):
        A, Q = np.diag([a, 0.5]), np.diag([0.0, 1.0])
        K, P, info = backend.dlqr(A, np.eye(2), Q, np.eye(2))
        assert info[0, 0] == ST_NOT_STABILISING, info
        assert np.isnan(K).all()
        assert np.isfinite(P).all() and P[0, 0, 0] == 0.0 and abs(P[0, 1, 1] - 1.1328) < 1e-4


def test_dlqr_uncontrollable_unstable_mode_is_nonfinite(backend):
    """A = diag(2, 0.5), B = [0; 1]: the unstable mode cannot be controlled (scipy raises LinAlgError).  H grows like
    4^(2^k) and overflows; that is -3 (non-finite), not a converged P = inf reported as -4 at the gain"""
    K, P, info = backend.dlqr(np.diag([2.0, 0.5]), np.array([[0.0], [1.0]]), np.eye(2), np.eye(1))
    assert info[0, 0] == ST_NONFINITE, info
    assert np.isnan(K).all()


def test_dlqr_singular_r_and_nonfinite_data(backend):
    r = np.random.default_rng(4)
    A, B = _systems(r, 3, 2, 0.8, 1)
    Q, R = _weights(r, 3, 2)
    K, _, info = backend.dlqr(A, B, Q, np.zeros((2, 2)))
    assert info[0, 0] == ST_R_SINGULAR and np.isnan(K).all()
    for what in ("A", "B", "Q", "R"):
        for bad in (np.nan, np.inf):
            a, b, q, rr = A.copy(), B.copy(), Q.copy(), R.copy()
            {"A": a[0], "B": b[0], "Q": q, "R": rr}[what][1, 0] = bad
            K, _, info = backend.dlqr(a, b, q, rr)
            assert info[0, 0] < 0 and np.isnan(K).all(), (what, bad, info)


def _doublings_scalar(a, q):
    """the doubling count of dlqr_one for A = [a], B = [0], Q = [q], R = [1], mirrored in double precision: G = 0 and
    W = 1, so every product the kernel forms is one correctly rounded multiplication"""
    h, ak = q, a
    for it in range(1, MAX_DOUBLINGS + 1):
        d = ak * (h * ak)
        h = h + d
        ak = ak * ak
        if abs(d) <= TOL * abs(h):
            return it
    return None


def test_dlqr_reports_the_doublings_done(backend):
    """info[:, 1] is the number of doublings done: exact against a mirror of the recurrence where it is exact"""
    a = np.array([0.0, 0.1, 0.5, -0.9, 0.99, 0.999999])
    K, P, info = backend.dlqr(a[:, None, None], np.zeros((a.size, 1, 1)), np.array([[2.0]]), np.array([[1.0]]))
    assert (info[:, 0] == ST_OK).all(), info
    assert info[:, 1].tolist() == [_doublings_scalar(x, 2.0) for x in a]
    assert np.allclose(P[:, 0, 0], 2.0 / (1 - a * a), rtol=1e-9, atol=0) and np.array_equal(K, np.zeros_like(K))


def test_dlqr_converging_on_the_last_allowed_doubling_is_converged():
    """host build only (max_doublings is not an argument of the C ABI): a system that meets the tolerance on exactly the
    last allowed doubling is converged (status 0), one doubling fewer is status 1 with every doubling counted"""
    h = HostLinalg()
    a = 0.99
    need = _doublings_scalar(a, 1.0)
    args = (np.array([[[a]]]), np.zeros((1, 1, 1)), np.array([[1.0]]), np.array([[1.0]]))
    _, _, info = h.dlqr(*args, max_doublings=need)
    assert info[0].tolist() == [ST_OK, need]
    K, _, info = h.dlqr(*args, max_doublings=need - 1)
    assert info[0].tolist() == [ST_NOT_CONVERGED, need - 1] and np.isfinite(K).all()


# ---------------------------------------------------------------------------------------------------------------------
# batch independence, reduced-model gather
# ---------------------------------------------------------------------------------------------------------------------
def test_failing_systems_do_not_touch_their_neighbours(backend):
    """a NaN system and a non-stabilising system in the middle of a batch: every other system's K, P, Ad, Bd are
    bit-identical to the same systems run as a batch without them"""
    r = np.random.default_rng(9)
    A, B = _systems(r, 2, 2, 1.1, 8)
    Q = np.diag([0.0, 1.0])  # shared: makes A = diag(1.5, 0.5) undetectable, the random systems are detectable
    bad_nan = np.full((1, 2, 2), np.nan)
    bad_und = np.diag([1.5, 0.5])[None]
    Ab = np.concatenate([A[:3], bad_nan, A[3:5], bad_und, A[5:]])
    Bb = np.concatenate([B[:3], np.eye(2)[None], B[3:5], np.eye(2)[None], B[5:]])
    keep = [0, 1, 2, 4, 5, 7, 8, 9]
    K0, P0, i0 = backend.dlqr(A, B, Q, np.eye(2))
    K1, P1, i1 = backend.dlqr(Ab, Bb, Q, np.eye(2))
    assert (i0[:, 0] == ST_OK).all() and i1[3, 0] < 0 and i1[6, 0] == ST_NOT_STABILISING
    assert np.array_equal(K1[keep], K0) and np.array_equal(P1[keep], P0) and np.array_equal(i1[keep], i0)
    Ad0, Bd0 = backend.zoh(A, B, 0.1)
    Ad1, Bd1 = backend.zoh(Ab * np.where(np.arange(10) == 6, 1e6, 1.0)[:, None, None], Bb, 0.1)  # and one that overflows
    assert np.isnan(Ad1[3]).all()
    assert np.array_equal(Ad1[keep], Ad0) and np.array_equal(Bd1[keep], Bd0)


def test_reduce_jacobian_is_the_gather(backend):
    """8192 random 18 x 18 Jacobians (the device kernel's grid-stride loop takes a second pass): bit-equal to
    A[:, NA_ROWS][:, :, NA_COLS] / NA_UCOLS"""
    A = np.random.default_rng(12).standard_normal((8192, 18, 18))
    Ana, Bna = backend.reduce_jacobian(A)
    assert np.array_equal(Ana, A[:, NA_ROWS][:, :, NA_COLS]) and np.array_equal(Bna, A[:, NA_ROWS][:, :, NA_UCOLS])


# ---------------------------------------------------------------------------------------------------------------------
# device only: grid-stride tails, device-buffer entry points, NULL outputs, argument checks, lqr_gain_batch
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_grid_stride_tails(f16):
    """N = 16 * 64 * sm_count + 37 2x1 systems: one more than a full grid of zoh / dlqr threads holds, so the last 37 are
    each a thread's second pass; they must be bit-equal to the same 37 run alone"""
    N = 16 * 64 * f16.lib.f16_sm_count() + 37
    r = np.random.default_rng(13)
    A, B = _systems(r, 2, 1, 0.95, N)
    Q, R = _weights(r, 2, 1)
    Ad, Bd = f16.discretise(A, B, 0.05)
    Ad1, Bd1 = f16.discretise(A[-37:], B[-37:], 0.05)
    assert np.array_equal(Ad[-37:], Ad1) and np.array_equal(Bd[-37:], Bd1)
    K, P, info = f16.dlqr(A, B, Q, R)
    K1, P1, info1 = f16.dlqr(A[-37:], B[-37:], Q, R)
    assert (info[:, 0] == ST_OK).all()
    assert np.array_equal(K[-37:], K1) and np.array_equal(P[-37:], P1) and np.array_equal(info[-37:], info1)


class _Dev:
    """device buffers through the library's allocator"""

    def __init__(self, f16):
        self.lib, self.ptrs = f16.lib, []

    def put(self, a):
        a = np.ascontiguousarray(a)
        p = self.lib.f16_dev_alloc(max(a.nbytes, 8))
        assert p
        self.ptrs.append(p)
        assert self.lib.f16_memcpy_h2d(p, _p(a), a.nbytes) == F16_OK
        return p

    def get(self, p, like):
        out = np.empty_like(like)
        assert self.lib.f16_memcpy_d2h(_p(out), p, out.nbytes) == F16_OK
        return out

    def free(self):
        for p in self.ptrs:
            self.lib.f16_dev_free(p)


@pytest.mark.gpu
def test_device_buffer_entry_points_equal_host_buffer_calls(f16):
    """discretise_batch_dev, dlqr_batch_dev (Q and R in device memory too), reduce_jacobian_batch_dev: bit-equal to the
    host-buffer calls on the same inputs"""
    r = np.random.default_rng(14)
    lib, dev = f16.lib, _Dev(f16)
    try:
        J = r.standard_normal((300, 18, 18))
        Ana, Bna = f16.reduce_jacobian(J)
        dA, dAna, dBna = dev.put(J), dev.put(np.zeros_like(Ana)), dev.put(np.zeros_like(Bna))
        assert lib.reduce_jacobian_batch_dev(dA, 300, dAna, dBna) == F16_OK
        assert np.array_equal(dev.get(dAna, Ana), Ana) and np.array_equal(dev.get(dBna, Bna), Bna)
        for n, m in ((9, 3), (18, 4), (1, 21), (5, 5)):
            A, B = _systems(r, n, m, 1.1, 50)
            Q, R = _weights(r, n, m)
            Ad, Bd = f16.discretise(A, B, 0.01)
            dA, dB, dAd, dBd = dev.put(A), dev.put(B), dev.put(np.zeros_like(A)), dev.put(np.zeros_like(B))
            assert lib.discretise_batch_dev(dA, dB, n, m, 50, 0.01, dAd, dBd) == F16_OK
            assert np.array_equal(dev.get(dAd, Ad), Ad) and np.array_equal(dev.get(dBd, Bd), Bd)
            K, P, info = f16.dlqr(Ad, Bd, Q, R)
            dQ, dR = dev.put(Q), dev.put(R)
            dK, dP, dI = dev.put(np.zeros_like(K)), dev.put(np.zeros_like(P)), dev.put(np.zeros_like(info))
            assert lib.dlqr_batch_dev(dAd, dBd, dQ, dR, n, m, 50, dK, dP, dI) == F16_OK
            assert np.array_equal(dev.get(dK, K), K) and np.array_equal(dev.get(dP, P), P)
            assert np.array_equal(dev.get(dI, info), info)
    finally:
        dev.free()


@pytest.mark.gpu
def test_dlqr_without_p_or_info(f16):
    """P = NULL and info = NULL leave K bit-unchanged"""
    r = np.random.default_rng(15)
    A, B = _systems(r, 6, 2, 1.2, 20)
    Q, R = _weights(r, 6, 2)
    K, P, info = f16.dlqr(A, B, Q, R)
    for with_p, with_info in ((False, True), (True, False), (False, False)):
        K1 = np.zeros_like(K)
        P1 = np.zeros_like(P) if with_p else None
        i1 = np.zeros_like(info) if with_info else None
        assert f16.lib.dlqr_batch(_p(A), _p(B), _p(Q), _p(R), 6, 2, 20, _p(K1), _p(P1), _p(i1)) == F16_OK
        assert np.array_equal(K1, K)
        assert P1 is None or np.array_equal(P1, P)
        assert i1 is None or np.array_equal(i1, info)


@pytest.mark.gpu
def test_argument_checks(f16):
    """bad shapes, NULL pointers with N > 0, a non-finite dt: F16_ERR_ARG with the outputs untouched; N = 0 is F16_OK"""
    lib = f16.lib
    N = 4
    big = np.zeros((N, 24, 24)) + 0.1
    sentinel = -12345.5

    def outs():
        return [np.full((N, 24, 24), sentinel), np.full((N, 24, 24), sentinel), np.full((N, 24, 24), sentinel),
                np.full((N, 2), 77, dtype=np.int32)]

    def untouched(o):
        return all((x == (77 if x.dtype == np.int32 else sentinel)).all() for x in o)

    dev = _Dev(f16)
    try:
        dbig = dev.put(big)
        for n, m in ((18, 5), (19, 1), (0, 1), (1, 0), (-1, 2), (4, -1)):
            o = outs()
            assert lib.discretise_batch(_p(big), _p(big), n, m, N, 0.01, _p(o[0]), _p(o[1])) == F16_ERR_ARG
            assert lib.dlqr_batch(_p(big), _p(big), _p(big), _p(big), n, m, N, _p(o[0]), _p(o[1]), _p(o[3])) == F16_ERR_ARG
            assert untouched(o), (n, m)
            do = [dev.put(x) for x in o]
            assert lib.discretise_batch_dev(dbig, dbig, n, m, N, 0.01, do[0], do[1]) == F16_ERR_ARG
            assert lib.dlqr_batch_dev(dbig, dbig, dbig, dbig, n, m, N, do[0], do[1], do[3]) == F16_ERR_ARG
            assert untouched([dev.get(p, x) for p, x in zip(do, o)]), (n, m)
        for dt in (np.nan, np.inf, -np.inf):
            o = outs()
            assert lib.discretise_batch(_p(big), _p(big), 3, 2, N, dt, _p(o[0]), _p(o[1])) == F16_ERR_ARG
            do = [dev.put(x) for x in o]
            assert lib.discretise_batch_dev(dbig, dbig, 3, 2, N, dt, do[0], do[1]) == F16_ERR_ARG
            assert untouched(o) and untouched([dev.get(p, x) for p, x in zip(do, o)]), dt
        o = outs()
        a, K = _p(big), _p(o[0])
        for args in ((None, a, 3, 2, N, 0.01, K, a), (a, None, 3, 2, N, 0.01, K, a), (a, a, 3, 2, N, 0.01, None, a),
                     (a, a, 3, 2, N, 0.01, K, None)):
            assert lib.discretise_batch(*args) == F16_ERR_ARG
        for i in range(5):  # Ad, Bd, Q, R, K
            args = [a, a, a, a, 3, 2, N, K, None, None]
            args[i if i < 4 else 7] = None
            assert lib.dlqr_batch(*args) == F16_ERR_ARG
        for args in ((None, N, K, K), (a, N, None, K), (a, N, K, None)):
            assert lib.reduce_jacobian_batch(*args) == F16_ERR_ARG
            assert lib.reduce_jacobian_batch_dev(*[dbig if x == a else x for x in args]) == F16_ERR_ARG
        assert untouched(o)
        assert lib.discretise_batch(a, a, 3, 2, -1, 0.01, K, K) == F16_ERR_ARG
        assert lib.dlqr_batch(a, a, a, a, 3, 2, -1, K, None, None) == F16_ERR_ARG
        assert lib.discretise_batch(None, None, 3, 2, 0, 0.01, None, None) == F16_OK
        assert lib.dlqr_batch(None, None, None, None, 3, 2, 0, None, None, None) == F16_OK
        assert lib.reduce_jacobian_batch(None, 0, None, None) == F16_OK
        assert lib.discretise_batch_dev(None, None, 3, 2, 0, 0.01, None, None) == F16_OK
        assert lib.dlqr_batch_dev(None, None, None, None, 3, 2, 0, None, None, None) == F16_OK
        assert lib.reduce_jacobian_batch_dev(None, 0, None, None) == F16_OK
    finally:
        dev.free()


@pytest.mark.gpu
def test_lqr_gain_batch_flags_an_out_of_envelope_point(f16):
    """perturbed trims of the golden xcg 0.35 aircraft plus one at alpha = 46 deg (outside the hifi tables): that point
    is flagged with NaN K; every other gain is bit-equal to the batch without it, and its closed loop is stable"""
    from _inputs import perturbed_trim
    g = load_golden("xcg35")
    x, u = perturbed_trim(12, g["x_trim"], seed=21, frac=0.01)
    xb = np.insert(x, 5, x[:, 0], axis=1)
    ub = np.insert(u, 5, u[:, 0], axis=1)
    xb[7, 5] = np.deg2rad(46.0)
    K0 = f16.F16Batch(x, u, xcg=0.35)._calc_LQR_gain()
    fb = f16.F16Batch(xb, ub, xcg=0.35)
    K1 = fb._calc_LQR_gain()
    assert fb.last_status[5] != 0 and np.isnan(K1[5]).all()
    assert (np.delete(fb.last_status, 5) == 0).all()
    assert np.array_equal(np.delete(K1, 5, axis=0), K0)
