"""Static split of an aircraft batch over the GPUs of one box (SURVEY.md 8e).

Aircraft never interact (env.py holds one state vector; Nlplant shares nothing but read-only tables), so the batch is
cut into contiguous slices of the aircraft axis, one per rank, and there is NO collective on the data path.  The
only communication is control-plane: a barrier around the timed region, the max-over-ranks duration, and one gather
of a small per-rank summary (survivors, per-state min / max / mean / M2).  `dist` is `torch.distributed` (NCCL on the
GPU box, gloo in the CPU tests) or None for a single process.
"""
import numpy as np


def shard_range(n_total, rank, world):
    """[lo, hi) of the aircraft axis owned by `rank`: contiguous, balanced to within one aircraft."""
    base, rem = divmod(int(n_total), int(world))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_soa(a, rank, world):
    """Slice of a [planes][N] SoA array owned by `rank` (C-contiguous copy, ready for the C ABI)."""
    lo, hi = shard_range(a.shape[-1], rank, world)
    return np.ascontiguousarray(a[..., lo:hi])


def rank_seed(seed, rank):
    """Per-rank RNG stream of the weak-scaling workloads (every rank draws its own aircraft)."""
    return int(seed) + int(rank)


def summarise(x, status):
    """Per-rank summary of a final state x [18][n]: [n, alive, then per state min, max, mean, M2 over survivors]."""
    alive = status == 0
    out = np.zeros(2 + 4 * 18)
    out[0], out[1] = x.shape[1], alive.sum()
    if alive.any():
        # C order, so the sums along each state run over contiguous memory and numpy sums them pairwise: the F-ordered copy
        # that x[:, alive] gives is summed one value after another, an error that grows with n (2300 ulp at 16 000 values)
        xa = np.ascontiguousarray(x[:, alive])
        mean = xa.mean(axis=1)
        out[2:20], out[20:38], out[38:56] = xa.min(axis=1), xa.max(axis=1), mean
        out[56:74] = ((xa - mean[:, None]) ** 2).sum(axis=1)
    else:
        out[2:20], out[20:38] = np.inf, -np.inf
    return out


def merge_summaries(rows):
    """Combine per-rank summaries (Chan et al. pairwise update of mean / M2)."""
    rows = np.asarray(rows, dtype=np.float64).reshape(-1, 74)
    n = rows[:, 0].sum()
    alive = rows[:, 1].sum()
    mn, mx = rows[:, 2:20].min(axis=0), rows[:, 20:38].max(axis=0)
    mean, m2 = np.zeros(18), np.zeros(18)
    cnt = 0.0
    for r in rows:
        k = r[1]
        if k == 0:
            continue
        d = r[38:56] - mean
        tot = cnt + k
        mean = mean + d * (k / tot)
        m2 = m2 + r[56:74] + d * d * (cnt * k / tot)
        cnt = tot
    return {"n": int(n), "alive": int(alive), "alive_fraction": float(alive / n) if n else 1.0,
            "min": mn, "max": mx, "mean": mean, "var": m2 / cnt if cnt else m2}


def max_over_ranks(dist, values, device="cpu"):
    """Element-wise max of a short list of floats over all ranks (timings are reported as the slowest rank's)."""
    if dist is None:
        return [float(v) for v in values]
    import torch
    t = torch.tensor(list(values), dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t.tolist()]


def gather_summaries(dist, row, device="cpu"):
    """All-gather of one per-rank summary row -> merged statistics (the only collective of a run)."""
    if dist is None:
        return merge_summaries([row])
    import torch
    t = torch.tensor(np.asarray(row, dtype=np.float64), device=device)
    out = [torch.zeros_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(out, t)
    return merge_summaries([o.cpu().numpy() for o in out])
