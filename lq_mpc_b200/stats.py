"""Column statistics of result tables, single- or multi-GPU.

The reference reduces every table over its sample axis with np.max / np.min / np.mean / np.std (utils.py:895-898).
Here each rank reduces its shard on the GPU in ONE pass (K5, csrc/k_stats.cu: max, min, counts, mean, M2 by
shifted-data accumulation with fixed-order folds) and the only data-path collective of the whole engine follows: one
all-gather of 6 doubles per column; every rank then merges the shards in rank order with Chan's pairwise update, so
all ranks hold bit-identical statistics and the result matches np.mean / np.std to rounding.

`merge_moments` is the pure host-side combination rule, shared by the NCCL path and the world_size-2 gloo tests.
`column_stats_two_pass` keeps np.std's literal two-pass scheme (three all-reduces) as a cross-check.

Order statistics over the same population (the entries with |x| <= 1.79e308, `k5_finite`; the moments' counts):
  * `column_quantiles`: exact np.quantile(..., method="linear"). The two order statistics each quantile interpolates
    between are selected on the GPU by radix descent (K5 `lqmpc_column_radix_histogram` / `_select`: 8 passes, one
    all-reduce of integer counts per pass when world > 1), and the interpolation runs on the host with numpy's own
    float64 operations, so the values equal numpy's (up to -0.0 standing for +0.0).
  * `column_argext`: max / min with the global index of the entry attaining them (ties: the lowest index), merged
    across ranks after one all-gather of (value, index) pairs.
"""
from __future__ import annotations

import math
from typing import Optional

import numpy as np


def finish(mx, mn, n_fin, n_bad, mean, m2):
    """Per-column dict in the reference's vocabulary from merged moments (numpy arrays)."""
    with np.errstate(invalid="ignore", divide="ignore"):
        std = np.sqrt(m2 / n_fin)
    return {"max": mx, "min": mn, "mean": mean, "std": std, "count": n_fin, "n_nonfinite": n_bad}


def merge_moments(parts):
    """Chan's pairwise update over shards, in shard (= rank) order. parts: [n_shards][cols][6] array with rows
    {max, min, n_finite, n_nonfinite, mean, M2}; empty shards (n_finite = 0) carry NaN mean/M2 and are skipped."""
    parts = np.asarray(parts, dtype=np.float64)
    cols = parts.shape[1]
    mx = np.full(cols, -np.inf); mn = np.full(cols, np.inf)
    n = np.zeros(cols); nb = np.zeros(cols); mean = np.zeros(cols); m2 = np.zeros(cols)
    for p in parts:
        bn = p[:, 2]
        has = bn > 0
        bmean = np.where(has, p[:, 4], 0.0)
        bm2 = np.where(has, p[:, 5], 0.0)
        tot = n + bn
        with np.errstate(invalid="ignore", divide="ignore"):
            w = np.where(tot > 0, bn / np.where(tot > 0, tot, 1.0), 0.0)
        delta = bmean - mean
        m2 = m2 + bm2 + delta * delta * n * w
        mean = mean + delta * w
        n = tot
        nb = nb + p[:, 3]
        mx = np.maximum(mx, p[:, 0]); mn = np.minimum(mn, p[:, 1])
    mean = np.where(n > 0, mean, np.nan)
    m2 = np.where(n > 0, m2, np.nan)
    return finish(mx, mn, n, nb, mean, m2)


def column_moments_device(engine, table, group=None):
    """Asynchronous half of `column_stats`: K5 on this rank's shard plus the all-gather, everything enqueued on the
    device; returns the [world][cols][6] DEVICE tensor of per-shard moments (no host synchronisation). Finish with
    `merge_moments(t.cpu().numpy())` whenever the numbers are needed on the host."""
    import torch
    import torch.distributed as dist
    mom = engine.column_moments_raw(table)                      # device [cols][6]
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        world = dist.get_world_size(group)
        allm = torch.empty((world,) + tuple(mom.shape), dtype=mom.dtype, device=mom.device)
        dist.all_gather_into_tensor(allm, mom, group=group)
        return allm
    return mom[None]


def column_stats(engine, table, group=None):
    """table: [cols][S_local] device tensor. One pass over the shard (K5 `lqmpc_column_moments`), ONE collective
    (all-gather of 6 doubles per column), Chan merge in rank order. Returns dict of numpy arrays (max, min, mean, std,
    count, n_nonfinite), identical on every rank."""
    return merge_moments(column_moments_device(engine, table, group).cpu().numpy())


def column_stats_two_pass(engine, table, group=None):
    """np.std's own two-pass scheme (max/min/sum/counts, all-reduce, squared deviations about the global mean,
    all-reduce): three collectives, two passes. Kept as the cross-check of the one-pass path."""
    import torch
    import torch.distributed as dist

    def _allreduce(t, op):
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            dist.all_reduce(t, op=op, group=group)
        return t
    raw = engine.column_stats_raw(table)                      # [cols][5]
    ext = torch.stack([raw[:, 0], -raw[:, 1]], dim=0).contiguous()
    add = torch.stack([raw[:, 2], raw[:, 3], raw[:, 4]], dim=0).contiguous()
    _allreduce(ext, dist.ReduceOp.MAX)
    _allreduce(add, dist.ReduceOp.SUM)
    mean = add[0] / add[1]
    sq = engine.column_sqdev_raw(table, mean)
    _allreduce(sq, dist.ReduceOp.SUM)
    return finish(ext[0].cpu().numpy(), -ext[1].cpu().numpy(), add[1].cpu().numpy(), add[2].cpu().numpy(),
                  mean.cpu().numpy(), sq.cpu().numpy())


# ---------------------------------------------------------------------------------------------------------------
# host-side protocol mirror (used by the gloo CPU tests: same collective and merge, partials supplied by the caller)
def local_moments_numpy(table):
    """What K5 (`moments_partial/final_kernel`) produces for one shard, restated with numpy for the CPU protocol tests
    only: [cols][6] = max, min, n_finite, n_nonfinite, mean, M2 with the same shifted-data formula."""
    t = np.asarray(table, dtype=np.float64)
    cols = t.shape[0]
    out = np.zeros((cols, 6))
    for c in range(cols):
        col = t[c]
        fin = np.isfinite(col)
        v = col[fin]
        k = col[0] if col.size and np.isfinite(col[0]) else 0.0
        n = float(v.size)
        d = v - k
        s1, s2 = d.sum(), (d * d).sum()
        out[c] = [v.max() if v.size else -np.inf, v.min() if v.size else np.inf, n, float((~fin).sum()),
                  k + s1 / n if n else np.nan, max(s2 - s1 * (s1 / n), 0.0) if n else np.nan]
    return out


def distributed_stats_protocol(local_table, group=None, partials=local_moments_numpy):
    """The one-collective protocol on CPU tensors (gloo). `local_table`: [cols][S_local] numpy array."""
    import torch
    import torch.distributed as dist
    mom = torch.from_numpy(np.ascontiguousarray(partials(local_table)))
    world = dist.get_world_size(group)
    gathered = [torch.empty_like(mom) for _ in range(world)]
    dist.all_gather(gathered, mom, group=group)
    return merge_moments(np.stack([g.numpy() for g in gathered]))


def shard_bounds(S: int, rank: int, world: int):
    """Contiguous shard [lo, hi) of the sample axis for `rank` (SURVEY 8e): sizes differ by at most one."""
    base, rem = divmod(S, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


# ---------------------------------------------------------------------------------------------------------------
# order statistics: exact quantiles (radix selection) and arg-extremes
FINITE_MAX = 1.79e308         # K5's population: |x| <= FINITE_MAX (csrc/k_stats.cu), also that of the moments
RADIX_MAX_SEL = 32            # selectors per histogram call (include/lqmpc_b200.h: LQMPC_RADIX_MAX_SEL)
_QS_PER_CALL = RADIX_MAX_SEL // 2   # two selectors per quantile: ranks floor(v) and floor(v) + 1


def k5_finite(x):
    """The entries K5 reduces: |x| <= 1.79e308. NaN and +-inf are out, and so are the few doubles above 1.79e308."""
    with np.errstate(invalid="ignore"):
        return np.abs(np.asarray(x, dtype=np.float64)) <= FINITE_MAX


def _world(group=None):
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size(group)
    return 1


def gather_rows(t, group=None):
    """[world] + t.shape: every rank's `t` in rank order (t[None] on one process)."""
    import torch
    import torch.distributed as dist
    world = _world(group)
    if world == 1:
        return t[None]
    if not t.is_cuda:
        parts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(parts, t.contiguous(), group=group)
        return torch.stack(parts)
    out = torch.empty((world,) + tuple(t.shape), dtype=t.dtype, device=t.device)
    dist.all_gather_into_tensor(out, t.contiguous(), group=group)
    return out


def check_quantiles(qs):
    """qs as a 1-D float64 array; ValueError unless every q is finite and in [0, 1]."""
    q = np.atleast_1d(np.asarray(qs, dtype=np.float64))
    if q.ndim != 1 or q.size == 0 or not np.all(np.isfinite(q)) or np.any(q < 0) or np.any(q > 1):
        raise ValueError("quantiles must be a non-empty list of finite numbers in [0, 1], got %r" % (qs,))
    return q


def radix_keys(x):
    """Order-preserving uint64 key of finite doubles: negatives get all bits flipped, non-negatives the sign bit set."""
    b = np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)
    return np.where(b >> np.uint64(63), ~b, b | np.uint64(1 << 63))


def keys_to_doubles(k):
    k = np.ascontiguousarray(k, dtype=np.uint64)
    return np.where(k >> np.uint64(63), k ^ np.uint64(1 << 63), ~k).view(np.float64)


def quantile_ranks(counts, qs):
    """numpy's neighbour indexes of the linear method (np.lib._function_base_impl._get_indexes) as 0-based ranks
    among the finite entries: torch int64 [cols][2 len(qs)] = (floor(v), floor(v) + 1) per q with v = (n - 1) q,
    both n - 1 where v >= n - 1. Computed where `counts` (float64 [cols]) lives, so no host read is needed."""
    import torch
    n = counts.to(torch.float64).reshape(-1, 1)
    q = torch.as_tensor(np.asarray(qs, dtype=np.float64), device=n.device).reshape(1, -1)
    v = (n - 1) * q
    last = (n - 1).expand_as(v)
    above = v >= last
    lo = torch.floor(v)
    r = torch.stack([torch.where(above, last, lo), torch.where(above, last, lo + 1)], dim=2)
    return r.reshape(n.shape[0], -1).clamp_min(0).to(torch.int64)


def radix_select_keys(counts, qs, histogram, reduce, select):
    """The selection protocol: per chunk of <= 16 quantiles, 8 x (histogram -> reduce -> select). `histogram(prefix,
    pass)` returns int64 [cols][nsel][256]; `reduce(hist)` sums it over ranks in place; `select(hist, pass, rank,
    prefix)` updates rank and prefix in place. Returns the keys, int64 [cols][2 len(qs)] (uint64 bit patterns)."""
    import torch
    keys = []
    for i in range(0, len(qs), _QS_PER_CALL):
        rank = quantile_ranks(counts, qs[i:i + _QS_PER_CALL])
        prefix = torch.zeros_like(rank)
        for p in range(8):
            h = histogram(prefix, p)
            reduce(h)
            select(h, p, rank, prefix)
        keys.append(prefix)
    return torch.cat(keys, dim=1)


def finish_quantiles(keys, counts, qs):
    """Host half: keys [cols][2 len(qs)] (uint64 or their int64 bit patterns), counts [cols] -> [len(qs)][cols]
    np.quantile values with numpy's own arithmetic (_get_indexes, _get_gamma, _lerp). NaN where a column has no finite
    entry."""
    qs = np.asarray(qs, dtype=np.float64)
    n = np.asarray(counts, dtype=np.float64)[None, :]
    x = keys_to_doubles(np.asarray(keys).view(np.uint64)).reshape(n.shape[1], len(qs), 2)
    a, b = x[:, :, 0].T, x[:, :, 1].T
    v = (n - 1) * qs[:, None]
    prev = np.where(v >= n - 1, -1.0, np.floor(v))
    gamma = v - prev
    with np.errstate(over="ignore", invalid="ignore"):
        diff = b - a
        res = a + diff * gamma
        res = np.where(gamma >= 0.5, b - diff * (1 - gamma), res)
    return np.where(n > 0, res, np.nan)


def _stage(engine, table):
    import torch
    with torch.cuda.stream(engine._stream):
        return engine._table_view(table)[0]


def column_quantile_keys(engine, table, qs, counts, group=None):
    """Device half of `column_quantiles`: the radix selection on this rank's shard, `counts` = the GLOBAL finite count
    per column (device float64 [cols]). Returns the device keys; nothing is read back."""
    import torch.distributed as dist

    def reduce(h):
        if _world(group) > 1:
            dist.all_reduce(h, op=dist.ReduceOp.SUM, group=group)
    return radix_select_keys(counts, check_quantiles(qs),
                             lambda prefix, p: engine.column_radix_histogram_raw(table, prefix, p), reduce,
                             engine.column_radix_select_raw)


def column_quantiles(engine, table, qs, group=None):
    """np.quantile(finite entries, q) for every q in qs and every column of a [cols][S_local] table (sharded over the
    ranks of `group` along the sample axis). Returns [len(qs)][cols], identical on every rank; NaN for a column without
    a finite entry. Collectives: the moments' all-gather (global counts) and one all-reduce per radix pass."""
    qs = check_quantiles(qs)
    t = _stage(engine, table)
    counts = column_moments_device(engine, t, group)[:, :, 2].sum(dim=0)
    keys = column_quantile_keys(engine, t, qs, counts, group)
    return finish_quantiles(keys.cpu().numpy(), counts.cpu().numpy(), qs)


def pack_argext(val, idx):
    """(val [cols][2], idx [cols][2]) -> int64 [cols][4] = {max bits, min bits, argmax, argmin}: one tensor to gather."""
    import torch
    return torch.cat([val.view(torch.int64), idx], dim=1)


def merge_argext(parts):
    """parts: [n_shards][cols][4] int64 packed (value, index) pairs in shard order. The largest (smallest) value
    wins; on ties the lowest index. Returns dict max, argmax, min, argmin (index -1 where no shard has a finite
    entry)."""
    parts = np.ascontiguousarray(parts, dtype=np.int64)
    vals = np.ascontiguousarray(parts[..., :2]).view(np.float64)
    idx = parts[..., 2:]
    cols = parts.shape[1]
    out = {}
    for j, (name, better) in enumerate((("max", np.greater), ("min", np.less))):
        best = np.full(cols, -np.inf if j == 0 else np.inf)
        arg = np.full(cols, -1, dtype=np.int64)
        for v, i in zip(vals[:, :, j], idx[:, :, j]):
            take = better(v, best) | ((v == best) & (i >= 0) & ((arg < 0) | (i < arg)))
            best = np.where(take, v, best)
            arg = np.where(take, i, arg)
        out[name], out["arg" + name] = best, arg
    return out


def default_index_base(S_local, group=None):
    """This rank's offset in the unsharded sample axis: the exclusive prefix sum of the ranks' lengths (one all-gather
    of one integer), which is `shard_bounds`' lo for contiguous shards."""
    import torch
    import torch.distributed as dist
    world = _world(group)
    if world == 1:
        return 0
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend(group) == "nccl" else "cpu"
    sizes = gather_rows(torch.tensor([int(S_local)], dtype=torch.int64, device=dev), group)
    return int(sizes[:dist.get_rank(group)].sum())


def column_argext_device(engine, table, group=None, index_base=None):
    """K5 arg-extremes of this rank's shard + the one all-gather; returns the device [world][cols][4] packed pairs."""
    t = _stage(engine, table)
    if index_base is None:
        index_base = default_index_base(t.shape[1], group)
    return gather_rows(pack_argext(*engine.column_argext_raw(t, index_base)), group)


def column_argext(engine, table, group=None, index_base=None):
    """Max / min of the finite entries of every column with the global index attaining them (ties: lowest index).
    Returns dict max, argmax, min, argmin (numpy [cols]), identical on every rank."""
    return merge_argext(column_argext_device(engine, table, group, index_base).cpu().numpy())


# host-side mirrors of the order-statistic kernels (CPU protocol tests only)
def radix_histogram_numpy(table, prefix, pass_):
    """What `lqmpc_column_radix_histogram` produces: int64 [cols][nsel][256]."""
    t = np.atleast_2d(np.asarray(table, dtype=np.float64))
    prefix = np.asarray(prefix).view(np.uint64)
    mask = np.uint64(0) if pass_ == 0 else np.uint64(((1 << 64) - 1) ^ ((1 << (64 - 8 * pass_)) - 1))
    hist = np.zeros(prefix.shape + (256,), dtype=np.int64)
    for c in range(t.shape[0]):
        k = radix_keys(t[c][k5_finite(t[c])])
        d = ((k >> np.uint64(56 - 8 * pass_)) & np.uint64(255)).astype(np.int64)
        for s in range(prefix.shape[1]):
            hist[c, s] = np.bincount(d[((k ^ prefix[c, s]) & mask) == 0], minlength=256)
    return hist


def radix_select_numpy(hist, pass_, rank, prefix):
    """What `lqmpc_column_radix_select` does, in place on rank (int64) and prefix (uint64 or int64 bit patterns)."""
    prefix = np.asarray(prefix).view(np.uint64)
    cum = np.cumsum(hist, axis=2)
    below = cum - hist
    inside = (rank[..., None] >= below) & (rank[..., None] < cum)
    found = inside.any(axis=2)
    d = inside.argmax(axis=2)
    rank[found] -= np.take_along_axis(below, d[..., None], axis=2)[..., 0][found]
    prefix[found] |= d[found].astype(np.uint64) << np.uint64(56 - 8 * pass_)


def distributed_quantiles_protocol(local_table, qs, group=None):
    """The quantile protocol on CPU tensors (gloo, or one process): numpy mirrors of the kernels, the same collectives
    and the same host finish as `column_quantiles`. `local_table`: [cols][S_local] numpy array."""
    import torch
    import torch.distributed as dist
    qs = check_quantiles(qs)
    t = np.atleast_2d(np.asarray(local_table, dtype=np.float64))
    counts = torch.from_numpy(k5_finite(t).sum(axis=1).astype(np.float64))

    def reduce(h):
        if _world(group) > 1:
            dist.all_reduce(h, op=dist.ReduceOp.SUM, group=group)
    reduce(counts)
    keys = radix_select_keys(counts, qs, lambda prefix, p: torch.from_numpy(radix_histogram_numpy(t, prefix.numpy(), p)),
                             reduce, lambda h, p, rank, prefix: radix_select_numpy(h.numpy(), p, rank.numpy(),
                                                                                   prefix.numpy()))
    return finish_quantiles(keys.numpy(), counts.numpy(), qs)


def local_argext_numpy(table, index_base=0):
    """What `lqmpc_column_argext` produces for one shard, packed as `pack_argext` packs it: int64 [cols][4]."""
    t = np.atleast_2d(np.asarray(table, dtype=np.float64))
    out = np.zeros((t.shape[0], 4), dtype=np.int64)
    vals = out[:, :2].copy().view(np.float64)
    for c in range(t.shape[0]):
        fin = np.flatnonzero(k5_finite(t[c]))
        if fin.size:
            v = t[c][fin]
            vals[c] = v.max(), v.min()
            out[c, 2:] = index_base + fin[np.argmax(v)], index_base + fin[np.argmin(v)]
        else:
            vals[c] = -np.inf, np.inf
            out[c, 2:] = -1
    out[:, :2] = vals.view(np.int64)
    return out


def distributed_argext_protocol(local_table, group=None, index_base=None):
    """The arg-extreme protocol on CPU tensors (gloo): default index base, one all-gather, merge in rank order."""
    import torch
    t = np.atleast_2d(np.asarray(local_table, dtype=np.float64))
    if index_base is None:
        index_base = default_index_base(t.shape[1], group)
    return merge_argext(gather_rows(torch.from_numpy(local_argext_numpy(t, index_base)), group).numpy())
