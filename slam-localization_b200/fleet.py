"""Host-side fleet logic for N > 1 GPUs: instance-index sharding and the end-of-run merge of the
ensemble statistics.  Filter instances share nothing (Usckf.hpp:77-78 / Msckf.hpp:74-75: every object
holds its state by value), so the step path has NO collective; the only exchange is one all-reduce of
`1 + N + N*N` doubles per fleet: (count, sum x, sum x x^T) as produced on each device by
slb_ensemble_stats (include/slb.h).  Backend-agnostic: NCCL on the GPUs, gloo in the CPU tests.
`consistency` turns the 6 sums of slb_consistency_stats / slb_gather_consistency into ANEES / ANIS and their chi-square
acceptance intervals."""
import math

import numpy as np


def shard_range(total, rank, world):
    """Contiguous shard [lo, hi) of `total` instances for `rank` of `world`; the remainder goes to the
    first ranks so shard sizes differ by at most one."""
    if not (0 <= rank < world) or total < 0:
        raise ValueError("bad shard request")
    base, rem = divmod(total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def stats_from_vectors(x):
    """(count, sum x, sum x x^T) flattened like slb_ensemble_stats, from vectorised means x[B, N]."""
    x = np.asarray(x, dtype=np.float64)
    n = x.shape[1]
    out = np.empty(1 + n + n * n)
    out[0] = x.shape[0]
    out[1:1 + n] = x.sum(axis=0)
    out[1 + n:] = (x.T @ x).ravel()
    return out


def merge_stats(stats, group=None):
    """All-reduce (SUM) a local statistics tensor in place across the process group and return it.
    A no-op when torch.distributed is not initialised (single GPU)."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=group)
    return stats


def make_nccl_comm(engine, rank, world):
    """An NCCL communicator for the C-level gather (slb_gather_stats): rank 0's unique id travels through the
    already-initialised torch.distributed group (any backend), every rank then joins through the C ABI."""
    import torch.distributed as dist

    def exchange(raw):
        box = [raw]
        dist.broadcast_object_list(box, src=0)
        return box[0]
    return engine.NcclComm(rank, world, exchange)


def moments(stats, n):
    """Ensemble mean and covariance from merged (count, sum x, sum x x^T)."""
    s = np.asarray(stats, dtype=np.float64)
    cnt = s[0]
    mean = s[1:1 + n] / cnt
    second = s[1 + n:].reshape(n, n) / cnt
    return cnt, mean, second - np.outer(mean, mean)


def _norm_ppf(p):
    """Standard normal quantile (Acklam's rational approximation refined by one Halley step on erfc: ~1e-15)."""
    a = (-3.969683028665376e+01, 2.209460984245205e+02, -2.759285104469687e+02, 1.383577518672690e+02,
         -3.066479806614716e+01, 2.506628277459239e+00)
    b = (-5.447609879822406e+01, 1.615858368580409e+02, -1.556989798598866e+02, 6.680131188771972e+01,
         -1.328068155288572e+01)
    c = (-7.784894002430293e-03, -3.223964580411365e-01, -2.400758277161838e+00, -2.549732539343734e+00,
         4.374664141464968e+00, 2.938163982698783e+00)
    d = (7.784695709041462e-03, 3.224671290700398e-01, 2.445134137142996e+00, 3.754408661907416e+00)
    if not 0.0 < p < 1.0:
        raise ValueError("p must lie in (0, 1)")
    if p < 0.02425 or p > 1 - 0.02425:
        q = math.sqrt(-2 * math.log(p if p < 0.5 else 1 - p))
        x = (((((c[0] * q + c[1]) * q + c[2]) * q + c[3]) * q + c[4]) * q + c[5]) / \
            ((((d[0] * q + d[1]) * q + d[2]) * q + d[3]) * q + 1)
        x = x if p < 0.5 else -x
    else:
        q = p - 0.5
        r = q * q
        x = (((((a[0] * r + a[1]) * r + a[2]) * r + a[3]) * r + a[4]) * r + a[5]) * q / \
            (((((b[0] * r + b[1]) * r + b[2]) * r + b[3]) * r + b[4]) * r + 1)
    e = 0.5 * math.erfc(-x / math.sqrt(2)) - p
    u = e * math.sqrt(2 * math.pi) * math.exp(x * x / 2)
    return x - u / (1 + x * u / 2)


def chi2_ppf(p, k):
    """Wilson-Hilferty approximation of the chi-square quantile with k degrees of freedom: k (1 - 2/(9k) + z sqrt(2/(9k)))^3
    with z the normal quantile of p (relative error below 1e-3 from k ~ 300 on, where fleet averages live)."""
    if k <= 0:
        raise ValueError("k must be positive")
    h = 2.0 / (9.0 * k)
    return k * max(1.0 - h + _norm_ppf(p) * math.sqrt(h), 0.0) ** 3


def consistency(stats, nees_dof, nis_dof, p=0.95):
    """ANEES / ANIS of slb_consistency_stats' 6 sums {NEES count, sum, sum of squares, NIS count, sum, sum of squares}
    (one 6-vector, or a list of per-step ones: summed, they give the time-averaged figures) and their two-sided
    acceptance intervals at probability p: a consistent filter's average of M chi-square(d) values lies in
    [chi2_{M d}((1 - p) / 2), chi2_{M d}((1 + p) / 2)] / M with probability p.  nees_dof / nis_dof: d of each, i.e. n of
    the NEES range and the measurement dimension.  An average over no instance is NaN with no interval."""
    s = np.asarray(stats, dtype=np.float64)
    if s.ndim == 2:
        s = s.sum(axis=0)
    if s.shape != (6,):
        raise ValueError("stats must be a 6-vector or a list of 6-vectors")
    out = {}
    for name, cnt, tot, dof in (("anees", s[0], s[1], nees_dof), ("anis", s[3], s[4], nis_dof)):
        m = int(round(cnt))
        out[name + "_count"] = m
        if m == 0 or dof <= 0:
            out[name], out[name + "_interval"] = float("nan"), None
            continue
        out[name] = tot / m
        out[name + "_interval"] = (chi2_ppf((1 - p) / 2, m * dof) / m, chi2_ppf((1 + p) / 2, m * dof) / m)
    return out
