"""The end-of-run statistics row [N, alive, min[18], max[18], mean[18], M2[18]] (csrc/f16_stats.cu, shard.summarise /
shard.merge_summaries) against an exact reference.

`exact_summary` is the row in exact arithmetic, rounded once: with fractions.Fraction for small selections, and for large ones
from error-free transformations (TwoSum deviations, Dekker products) summed by math.fsum.  The second form is checked against
the first before anything is checked against it.

The kernel folds S1 = sum (v - c), S2 = sum (v - c)^2 with c = the first survivor's state, over a fixed tree: a thread's
grid-stride run, five warp shuffles, eight warps in shared memory, then the finishing CTA's lanes over the per-CTA partials and
five more shuffles.  Each value meets at most `depth` additions, so with eps = 2^-52
    mean:  |m - mu|   <= 4 ulp(mu) + A eps mean|v - c|
    M2:    |M2 - M2*| <= B eps (M2* + n (mu - c)^2)          (S2 carries depth eps S2; S1^2 / n twice the error of S1)
with A = depth + 4 and B = 3 A at the largest batch tested (2^22 + 3 aircraft, about 37 per thread at 148 SMs).  The shift
enters the bar: a shift far outside the survivors inflates both bars, and the shift the kernel may use is the first
survivor's, nothing else.  Counts, min and max are exact.

Worst error as a fraction of its bar, measured on an NVIDIA B200 (1000 W power limit), A = 72, B = 216:
    one context, every size and mask           mean 0.25    M2 0.0072
    the outlier plane (first survivor 1e3 sigma out)  mean 0.011   M2 0.0084  (about 4e-10 of M2)
    rollout_stats, fast and strict             mean 0.017   M2 0.0064
    2 and 3 contexts (Chan's update included)  mean 0.25    M2 0.046
The mean's 0.25 is one ulp against a bar of four on a plane whose mean lies near the shift.  A dead aircraft's NaN, infinity
or 1e300 reaching a sum leaves a non-finite or far-off field where the exact one is finite: check_row counts a NaN as a
failure."""
import ctypes
import importlib.util
import math
import os
from fractions import Fraction

import numpy as np
import pytest

EPS = np.finfo(np.float64).eps
INT_MIN, INT_MAX = -2**31, 2**31 - 1
FRACTION_BELOW = 4096      # selections up to this size get the Fraction reference

# the sharding module alone (as tests/test_multirank.py loads it): the CPU tests need no built library
_spec = importlib.util.spec_from_file_location(
    "shard", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "f16_mpc_oop_py_b200", "shard.py"))
shard = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(shard)


# ---------------------------------------------------------------------------------------------------------
# the exact reference
# ---------------------------------------------------------------------------------------------------------
def _two_sum(a, b):
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def _split(a):
    t = 134217729.0 * a      # 2^27 + 1
    hi = t - (t - a)
    return hi, a - hi


def _two_prod(a, b):
    p = a * b
    ah, al = _split(a)
    bh, bl = _split(b)
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


def _plane_fraction(v):
    fr = [Fraction(float(t)) for t in v]
    mu = sum(fr) / len(fr)
    return float(mu), float(sum((t - mu) ** 2 for t in fr))


def _plane_fsum(v):
    """mean and M2 of finite values: m0 = fsum / n, D = sum (v - m0) exactly, mean = m0 + D / n, and
    M2 = sum (v - m0)^2 - D^2 / n with (v - m0) = hi + lo and (v - m0)^2 = hi^2 + 2 hi lo + lo^2, hi^2 and hi lo as exact
    products (lo^2 alone is rounded: it is below eps^2 of its term)."""
    n = v.size
    m0 = math.fsum(v.tolist()) / n
    with np.errstate(all="ignore"):
        hi, lo = _two_sum(v, -m0)
        d = math.fsum(np.concatenate([hi, lo]).tolist())
        p, e = _two_prod(hi, hi)
        q, f = _two_prod(hi, lo)
        s = math.fsum(np.concatenate([p, e, 2 * q, 2 * f, lo * lo]).tolist() + [-(d * d) / n])
    return m0 + d / n, max(s, 0.0)


def exact_summary(x, status=None, fraction_below=FRACTION_BELOW):
    """The 74-double row over the aircraft with status 0 (all of them for status None), each field rounded once from its exact
    value.  A survivor's NaN or infinity, per plane: min / max skip a NaN; M2 is NaN; the mean is NaN when the plane holds a
    NaN or both infinities, else that infinity (include/f16_b200.h)."""
    x = np.asarray(x, dtype=np.float64)
    n = x.shape[1]
    alive = np.ones(n, bool) if status is None else np.asarray(status) == 0
    k = int(alive.sum())
    row = np.zeros(74)
    row[0], row[1] = n, k
    row[2:20], row[20:38] = np.inf, -np.inf
    if k == 0:
        return row
    for i in range(18):
        v = x[i, alive]
        nn = v[~np.isnan(v)]
        if nn.size:
            row[2 + i], row[20 + i] = nn.min(), nn.max()
        if not np.isfinite(v).all():
            pos, neg = (v == np.inf).any(), (v == -np.inf).any()
            row[38 + i] = np.nan if np.isnan(v).any() or (pos and neg) else (np.inf if pos else -np.inf)
            row[56 + i] = np.nan
            continue
        row[38 + i], row[56 + i] = _plane_fraction(v) if k <= fraction_below else _plane_fsum(v)
    return row


# ---------------------------------------------------------------------------------------------------------
# test data: eighteen planes of different designs, masks that put the survivors where the kernel's arithmetic depends on it
# ---------------------------------------------------------------------------------------------------------
OUTLIER = 6        # the plane whose first survivor sits 1e3 standard deviations out (the documented limit of the shift)
POISON = (np.nan, np.inf, -np.inf, 1e300, -1e300)


def planes(n, seed):
    r = np.random.default_rng(seed)
    z, u = r.standard_normal, r.uniform
    x = np.empty((18, n))
    x[0] = u(-1e4, 1e4, n)                       # uniform +-1e4
    x[1] = 1e4 + 1e-3 * z(n)                     # narrow: sum-of-squares forms cancel
    x[2] = 1e8 + z(n)                            # offset
    x[3] = 1234.5678901234567                    # constant: M2 exactly 0, mean exactly the value
    x[4] = 1e-150 * (1 + 0.5 * u(-1, 1, n))      # tiny, squares still normal
    x[5] = z(n)                                  # mixed signs about 0
    x[6] = 5 + 1e-2 * z(n)                       # OUTLIER (its first survivor is set by with_mask)
    x[7] = -1e4 + 1e-3 * z(n)
    x[8] = 1e-150 * z(n)                         # tiny, mixed signs
    x[9] = -1e8 + z(n)
    x[10] = -0.1                                 # constant, negative
    x[11] = 3e5 + 1e-2 * u(-1, 1, n)
    x[12] = u(-1, 1, n)
    x[13] = 1e4 + z(n)
    x[14] = 1e-3 * z(n)
    x[15] = np.sign(z(n)) * 10.0 ** u(-5, 5, n)  # ten decades
    x[16] = 700 + 35 * u(-1, 1, n)
    x[17] = u(-1e12, 1e12, n)
    return x


def with_mask(x, status):
    """x with every dead aircraft carrying NaN, +-inf or +-1e300 in every plane, and the outlier plane's first survivor
    1e3 standard deviations out"""
    x = x.copy()
    alive = np.ones(x.shape[1], bool) if status is None else status == 0
    dead = np.flatnonzero(~alive)
    x[:, dead] = np.array(POISON)[np.arange(dead.size) % len(POISON)]
    if alive.any():
        x[OUTLIER, np.argmax(alive)] = 5 + 1e3 * 1e-2
    return x


def masks(n, seed):
    """name -> status [n] int32 (None: no status array)"""
    r = np.random.default_rng(seed)
    out = {"none": None, "zeros": np.zeros(n, np.int32)}
    st = np.where(r.uniform(size=n) < 0.2, r.choice([1, 4, -1, INT_MIN, INT_MAX, 1 << 18], n), 0).astype(np.int32)
    out["random20"] = st
    out["all_dead"] = np.full(n, 4, np.int32)
    for j in (0, 31, 32, 33, n - 1):
        if 0 <= j < n:
            s = r.choice([1, -7, INT_MIN, INT_MAX], n).astype(np.int32)
            s[j] = 0
            out[f"one_at_{j}"] = s
    for k in (1, 3, 40):
        if 32 * k < n:
            s = st.copy()
            s[:32 * k] = r.choice([2, -2, INT_MIN], 32 * k)
            out[f"first_{32 * k}_dead"] = s
    return out


# ---------------------------------------------------------------------------------------------------------
# bars
# ---------------------------------------------------------------------------------------------------------
def tree_depth(n, sm_count):
    """additions a value meets on its way to S1 / S2 (csrc/f16_stats.cu: grid = min(ceil(n / 256), 3 SMs) CTAs of 256)"""
    grid = max(1, min(-(-n // 256), 3 * sm_count))
    return -(-n // (grid * 256)) + 5 + 7 + -(-grid // 32) + 5


def shift_terms(x, alive, spans):
    """per plane over the slices `spans` [(lo, n)]: sum |v - c|, sum_k n_k (mean_k - c_k)^2 with c_k the first survivor of
    slice k (0 for a non-finite value, as the kernel takes it), and sum_k n_k (mean_k - mean)^2 (the spread between slices)"""
    dev, off, means, counts = np.zeros(18), np.zeros(18), [], []
    for lo, m in spans:
        a = alive[lo:lo + m]
        if not a.any():
            continue
        v = x[:, lo:lo + m][:, a]
        c = v[:, 0].copy()
        c[~np.isfinite(c)] = 0.0
        d = v - c[:, None]
        dev += np.abs(d).sum(axis=1)
        off += v.shape[1] * d.mean(axis=1) ** 2
        means.append(v.mean(axis=1))
        counts.append(v.shape[1])
    means, counts = np.array(means), np.array(counts, float)[:, None]
    mean = (means * counts).sum(axis=0) / counts.sum()
    return dev, off, (counts * (means - mean) ** 2).sum(axis=0)


def check_row(row, ref, x, status, A, B, spans=None):
    """row against exact_summary's ref; returns each plane's error as a fraction of its bar, (mean[18], M2[18]).  The rows of several
    slices are merged on the host by Chan's update (merge_summary_row), which is first order in the rounding of the slice
    means: a slice mean off by delta moves the term d^2 n_a n_b / n of M2 by 2 |d| delta n_a n_b / n.  So a merged row's M2
    gets 4 delta sqrt(k S) + 4 k delta^2 more, S the spread between the slices (Cauchy-Schwarz) and delta the mean bar."""
    n = x.shape[1]
    alive = np.ones(n, bool) if status is None else np.asarray(status) == 0
    assert row[0] == ref[0] and row[1] == ref[1], (row[:2], ref[:2])
    assert np.array_equal(row[2:38], ref[2:38]), "min / max"
    k = ref[1]
    if k == 0:
        assert not row[38:].any()
        return np.zeros(18), np.zeros(18)
    fin = np.isfinite(ref[38:56]) & np.isfinite(ref[56:74])
    assert np.array_equal(row[38:74][~np.tile(fin, 2)], ref[38:74][~np.tile(fin, 2)], equal_nan=True), "non-finite fields"
    spans = spans or [(0, n)]
    with np.errstate(all="ignore"):
        dev, off, between = shift_terms(np.where(np.isfinite(x), x, 0.0), alive, spans)
        mu, m2 = ref[38:56], ref[56:74]
        bar_m = 4 * np.spacing(np.abs(mu)) + A * EPS * dev / k
        bar_2 = B * EPS * (m2 + off)
        if len(spans) > 1:
            bar_2 = bar_2 + 4 * bar_m * np.sqrt(k * between) + 4 * k * bar_m ** 2
        em, e2 = np.abs(row[38:56] - mu), np.abs(row[56:74] - m2)
        bad = fin & ~((em <= bar_m) & (e2 <= bar_2))       # a NaN where the exact value is finite fails
        assert not bad.any(), [(i, row[38 + i], mu[i], bar_m[i], row[56 + i], m2[i], bar_2[i]) for i in np.flatnonzero(bad)]
        fm = np.where(fin & (bar_m > 0), em / bar_m, 0.0)
        f2 = np.where(fin & (bar_2 > 0), e2 / bar_2, 0.0)
    return fm, f2


def _report(what, fractions, outlier=True):
    """print the worst error / bar of a test (pytest -s shows it), the outlier plane of `planes` apart"""
    fm = np.max([f[0] for f in fractions], axis=0)
    f2 = np.max([f[1] for f in fractions], axis=0)
    rest = np.arange(18) != OUTLIER if outlier else np.ones(18, bool)
    line = f"{what}: worst error / bar  mean {fm[rest].max():.3g}  M2 {f2[rest].max():.3g}"
    if outlier:
        line += f";  outlier plane  mean {fm[OUTLIER]:.3g}  M2 {f2[OUTLIER]:.3g}"
    print(line)


# ---------------------------------------------------------------------------------------------------------
# CPU: the reference itself, and shard.summarise / merge_summaries
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 2, 3, 31, 33, 257, 1000])
def test_fsum_reference_agrees_with_fractions(n):
    """the large-N form of exact_summary within 1 ulp of the Fraction form, every plane and mask"""
    x = planes(n, seed=n)
    for name, st in masks(n, seed=n + 1).items():
        xm = with_mask(x, st)
        a = exact_summary(xm, st)
        b = exact_summary(xm, st, fraction_below=0)
        assert np.array_equal(a[:38], b[:38]), name
        assert np.all(np.abs(a[38:] - b[38:]) <= np.spacing(np.abs(a[38:]))), (name, np.flatnonzero(a[38:] != b[38:]))


def test_exact_reference_edges():
    x = planes(5, seed=1)
    st = np.array([3, 0, -1, 0, INT_MIN], np.int32)
    xm = with_mask(x, st)
    ref = exact_summary(xm, st)
    assert ref[0] == 5 and ref[1] == 2 and ref[38 + 3] == x[3, 0] and ref[56 + 3] == 0.0 and ref[56 + 10] == 0.0
    v = xm[:, [1, 3]]
    assert np.array_equal(ref[2:20], v.min(axis=1)) and np.array_equal(ref[20:38], v.max(axis=1))
    one = exact_summary(xm[:, 1:2])
    assert np.array_equal(one[38:56], xm[:, 1]) and not one[56:].any()
    # a survivor's non-finite values (status None): min / max skip NaN, M2 NaN, mean NaN or the infinity
    y = planes(6, seed=2)
    y[0, 2], y[1, 3], y[2, 1], y[2, 4], y[3, 0] = np.nan, np.inf, np.inf, -np.inf, -np.inf
    r = exact_summary(y)
    assert np.isnan(r[38]) and r[39] == np.inf and np.isnan(r[40]) and r[41] == -np.inf and np.isnan(r[56:60]).all()
    assert r[2] == np.nanmin(y[0]) and r[21] == np.inf and r[2 + 3] == -np.inf and np.isfinite(r[38 + 4:56]).all()


def _split_rows(x, st, cuts):
    edges = [0] + sorted(cuts) + [x.shape[1]]
    return [shard.summarise(x[:, lo:hi], st[lo:hi]) for lo, hi in zip(edges[:-1], edges[1:]) if hi > lo]


@pytest.mark.parametrize("seed", range(6))
def test_summarise_and_merge_against_exact(seed):
    """shard.summarise per rank, shard.merge_summaries over 1 to 8 ranks, against the exact row of the whole batch.
    Each rank's mean is numpy's pairwise sum over n (error below 32 eps max|v|, delta); Chan's update is first order in
    those errors, so
        mean:  |m - mu|            <= 4 ulp(mu) + delta
        var:   |var - M2* / k| k   <= 64 eps M2* + 4 delta sqrt(k M2*) + 4 k delta^2
    Ranks with no survivor and with exactly one are in every split."""
    r = np.random.default_rng(100 + seed)
    n = 20_000
    x = planes(n, seed=seed)
    st = np.where(r.uniform(size=n) < 0.2, 4, 0).astype(np.int32)
    ranks = int(r.integers(1, 9))
    cuts = list(r.choice(np.arange(1, n - 200), ranks - 1, replace=False))
    if ranks >= 3:                                   # one rank with no survivor, one with exactly one
        a, b = int(r.integers(1, n // 2 - 100)), int(r.integers(n // 2, n - 200))
        st[a:a + 50] = 4
        st[b:b + 50] = 4
        st[b + 17] = 0
        cuts = sorted(set(cuts[:ranks - 3]) | {a, a + 50, b, b + 50})
    x = with_mask(x, st)
    ref = exact_summary(x, st)
    merged = shard.merge_summaries(_split_rows(x, st, cuts))
    k = ref[1]
    assert merged["n"] == n and merged["alive"] == k
    assert np.array_equal(merged["min"], ref[2:20]) and np.array_equal(merged["max"], ref[20:38])
    vmax = np.abs(x[:, st == 0]).max(axis=1)
    delta = 32 * EPS * vmax
    mu, m2 = ref[38:56], ref[56:74]
    assert np.all(np.abs(merged["mean"] - mu) <= 4 * np.spacing(np.abs(mu)) + delta)
    err = np.abs(merged["var"] * k - m2)
    assert np.all(err <= 64 * EPS * m2 + 4 * delta * np.sqrt(k * m2) + 4 * k * delta ** 2), err / np.maximum(m2, 1e-300)


def test_merge_of_empty_and_single_survivor_ranks():
    x = planes(96, seed=9)
    st = np.full(96, 1, np.int32)
    st[70] = 0
    x = with_mask(x, st)
    ref = exact_summary(x, st)
    merged = shard.merge_summaries(_split_rows(x, st, [32, 64]))
    assert merged["alive"] == 1 and np.array_equal(merged["mean"], ref[38:56]) and not merged["var"].any()
    none = shard.merge_summaries(_split_rows(x, np.ones(96, np.int32), [10, 50]))
    assert none["alive"] == 0 and np.all(np.isposinf(none["min"])) and not none["mean"].any()


# ---------------------------------------------------------------------------------------------------------
# GPU: the device row against the exact one
# ---------------------------------------------------------------------------------------------------------
LARGEST = (1 << 22) + 3       # every thread folds about 37 aircraft at 148 SMs


def _bars(f16):
    d = tree_depth(LARGEST, f16.lib.f16_sm_count())
    return d + 4, 3 * (d + 4)


def _sizes(sm_count):
    cap = 3 * sm_count * 256      # aircraft the grid covers in one sweep
    return [1, 2, 31, 32, 33, 255, 256, 257, 8191, 8193, cap - 1, cap + 1, LARGEST]


class _Dev:
    """device copies of x (plane stride ld, NaN in the padding) and of the status words"""

    def __init__(self, f16, x, status, pad=0):
        L = f16.lib
        self.L, n = L, x.shape[1]
        self.ld = n + pad
        X = np.full((18, self.ld), np.nan)
        X[:, :n] = x
        self.d_x = L.f16_dev_alloc(X.nbytes)
        assert self.d_x and L.f16_memcpy_h2d(self.d_x, X.ctypes.data, X.nbytes) == 0
        self.d_st = None
        if status is not None:
            st = np.ascontiguousarray(status, np.int32)
            self.d_st = L.f16_dev_alloc(max(st.nbytes, 4))
            assert self.d_st and L.f16_memcpy_h2d(self.d_st, st.ctypes.data, st.nbytes) == 0

    def free(self):
        for p in (self.d_x, self.d_st):
            if p:
                self.L.f16_dev_free(p)


def _size_ids():
    return ["1", "2", "31", "32", "33", "255", "256", "257", "8191", "8193", "cap-1", "cap+1", "largest"]


@pytest.mark.gpu
@pytest.mark.parametrize("which", range(13), ids=_size_ids())
def test_state_summary_against_exact(f16, which):
    """every mask at every size (the 2^22 + 3 batch: the masks that matter for the shift, and one survivor), host and device
    entry points; the device call with plane stride ld > N and NaN in the padding"""
    sm = f16.lib.f16_sm_count()
    n = _sizes(sm)[which]
    A, B = _bars(f16)
    x0 = planes(n, seed=n)
    all_masks = masks(n, seed=n + 1)
    if n == LARGEST:
        all_masks = {k: v for k, v in all_masks.items() if k in ("none", "zeros", "first_1280_dead", f"one_at_{n - 1}", "all_dead")}
    worst, rows, refs = [], {}, {}
    for name, st in all_masks.items():
        x = with_mask(x0, st)
        ref = refs["none"] if name == "zeros" else exact_summary(x, st)        # the same selection and values
        refs[name] = ref
        row = f16.state_summary(x, st)
        worst.append(check_row(row, ref, x, st, A, B))
        rows[name] = row
        dev = _Dev(f16, x, st, pad=3 if n % 2 else 64)
        try:
            rd = f16.state_summary_dev(dev.d_x, dev.ld, n, dev.d_st)
            assert np.array_equal(rd, row, equal_nan=True), name                   # host and device entry points
            assert np.array_equal(f16.state_summary_dev(dev.d_x, dev.ld, n, dev.d_st), rd, equal_nan=True), name
        finally:
            dev.free()
    assert np.array_equal(rows["none"], rows["zeros"])                             # no status array = all zeros, same bits
    _report(f"state_summary n={n}", worst)


@pytest.mark.gpu
def test_state_summary_survivors_with_non_finite_values(f16):
    """status None: a survivor's NaN / infinity is a value like any other, and the row reports it as the header says"""
    n = 5000
    A, B = _bars(f16)
    x = planes(n, seed=77)
    x[0, 40], x[1, 0], x[2, 100], x[2, 4000], x[5, 4999], x[12, 7] = np.nan, np.inf, np.inf, -np.inf, -np.inf, np.nan
    x[12, 9] = np.inf
    ref = exact_summary(x)
    assert np.isnan(ref[38]) and ref[39] == np.inf and np.isnan(ref[40]) and ref[43] == -np.inf
    check_row(f16.state_summary(x), ref, x, None, A, B)
    dev = _Dev(f16, x, None, pad=5)
    try:
        check_row(f16.state_summary_dev(dev.d_x, dev.ld, n, None), ref, x, None, A, B)
    finally:
        dev.free()


def _slices(f16, n, min_per_device, contexts):
    lo_n = (ctypes.c_longlong * (2 * contexts))()
    k = f16.lib.f16_plan_slices(n, min_per_device, contexts, lo_n)
    return [(lo_n[2 * i], lo_n[2 * i + 1]) for i in range(k)]


# minimum slice sizes of the sliced calls (f16_api.cu: state_summary_batch 65536, step_batch_stats 16384 aircraft per context)
SUMMARY_SLICE, STATS_SLICE = 65536, 16384


def _open_loop_batch(n, seed):
    """xcg 0.35 open loop about trim, +-5 %: casualties accumulate; the first 40 aircraft start below the ground"""
    from _inputs import perturbed_trim
    from conftest import load_golden
    x, u = perturbed_trim(n, load_golden("xcg35")["x_trim"], seed=seed, frac=0.05)
    x[2, :40] = -1.0
    return x, u


@pytest.mark.gpu
@pytest.mark.parametrize("contexts", [2, 3])
def test_slices_over_contexts_against_exact(f16, contexts):
    """state_summary_batch and step_batch_stats over 2 and 3 contexts of one GPU: each slice takes its own shift, and the second
    slice starts with 32 dead aircraft; the merged rows against the exact rows"""
    A, B = _bars(f16)
    try:
        f16.shutdown()
        assert f16.init_devices([0] * contexts) == contexts
        n = 3 * SUMMARY_SLICE + 1001
        spans = _slices(f16, n, SUMMARY_SLICE, contexts)
        assert len(spans) == contexts
        x0 = planes(n, seed=contexts)
        st = masks(n, seed=5)["random20"]
        st[spans[1][0]:spans[1][0] + 32] = INT_MIN
        x = with_mask(x0, st)
        _report(f"state_summary over {contexts} contexts",
                [check_row(f16.state_summary(x, st), exact_summary(x, st), x, st, A, B, spans=spans)])

        n, K, M = 3 * STATS_SLICE + 501, 600, 150
        spans = _slices(f16, n, STATS_SLICE, contexts)
        assert len(spans) == contexts
        x, u = _open_loop_batch(n, seed=21)
        x[2, spans[1][0]:spans[1][0] + 32] = -1.0
        rows = f16.F16Batch(x, u, xcg=0.35).rollout_stats(K, M)
        b = f16.F16Batch(x, u, xcg=0.35)
        worst = []
        for i in range(K // M):
            b.step(K=M)
            assert np.all(b.status[:40] != 0) and np.all(b.status[spans[1][0]:spans[1][0] + 32] != 0)
            worst.append(check_row(rows[i], exact_summary(b.x, b.status), b.x, b.status, A, B, spans=spans))
        _report(f"step_batch_stats over {contexts} contexts", worst, outlier=False)
    finally:
        f16.shutdown()
        f16.init()


@pytest.mark.gpu
@pytest.mark.parametrize("math", ["fast", "strict"])
def test_rollout_stats_against_exact(f16, math):
    """F16Batch.rollout_stats, one context: every snapshot row against the exact row of the states and status words that
    repeated step(M) calls give (test_gpu_parity.py shows those are the snapshot's bits); the first survivor moves as
    aircraft die, so every row takes a new shift"""
    A, B = _bars(f16)
    prev = f16.lib.f16_set_math_mode(f16.MATH_FAST if math == "fast" else f16.MATH_STRICT)
    try:
        n, K, M = 20_000, 3000, 375
        x, u = _open_loop_batch(n, seed=31)
        rows = f16.F16Batch(x, u, xcg=0.35).rollout_stats(K, M)
        b = f16.F16Batch(x, u, xcg=0.35)
        worst = []
        for i in range(K // M):
            b.step(K=M)
            assert np.all(b.status[:40] != 0)
            worst.append(check_row(rows[i], exact_summary(b.x, b.status), b.x, b.status, A, B))
        _report(f"rollout_stats {math}", worst, outlier=False)
        assert rows[-1][1] <= rows[0][1] <= n - 40
    finally:
        f16.lib.f16_set_math_mode(prev)
