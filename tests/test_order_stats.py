"""CPU tier — exact column quantiles and arg-extremes: the numpy restatement of the radix-selection kernels and the
host finish give np.quantile's values exactly on adversarial columns, and the gloo protocol on uneven shards (world
sizes 2 and 3) equals the single-shard result bit for bit."""
import os
import socket

import numpy as np
import pytest

from lq_mpc_b200 import stats as st

QS = [0.0, 1.0, 0.5, 1 / 3, 0.999999, 0.25, 0.75, 0.05, 0.95]


def adversarial_columns():
    """Named 1-D columns: ties, all-equal, signed zeros, subnormals, +-1e308, mixed NaN / +-inf, n = 0, 1, 2."""
    rng = np.random.default_rng(11)
    mixed = rng.normal(size=301)
    mixed[::7] = np.nan
    mixed[::11] = np.inf
    mixed[::13] = -np.inf
    return {
        "normal": rng.normal(size=1001),
        "ties": rng.integers(-2, 3, size=777).astype(np.float64),
        "all_equal": np.full(64, 0.1),
        "signed_zeros": np.array([0.0, -0.0, 0.0, -0.0, 1.0, -1.0, -0.0]),
        "subnormals": np.array([5e-324, -5e-324, 2.2e-308, -2.2e-308, 1e-310, 0.0, -1e-310, 3e-320]),
        "huge": np.array([1e308, -1e308, 1.7976931348623157e308, -1.7976931348623157e308, 1.0, 0.0]),
        "mixed_nonfinite": mixed,
        "all_nonfinite": np.array([np.nan, np.inf, -np.inf, np.nan]),
        "n0": np.array([]),
        "n1": np.array([2.5]),
        "n2": np.array([3.0, -1.0]),
        "n2_equal": np.array([-7.0, -7.0]),
    }


def _np_quantile(col, qs):
    f = col[st.k5_finite(col)]
    if f.size == 0:
        return np.full(len(qs), np.nan)
    with np.errstate(over="ignore", invalid="ignore"):
        return np.quantile(f, qs)


def _same(a, b):
    """Value-equal, NaN == NaN; -0.0 and +0.0 may stand for each other."""
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and bool(np.all((a == b) | (np.isnan(a) & np.isnan(b))))


def test_key_map_is_order_preserving_and_invertible():
    rng = np.random.default_rng(1)
    x = np.concatenate([rng.normal(size=1000) * 10.0 ** rng.integers(-300, 300, size=1000),
                        [0.0, -0.0, 5e-324, -5e-324, 1.7976931348623157e308, -1.7976931348623157e308]])
    k = st.radix_keys(x)
    assert np.array_equal(st.keys_to_doubles(k).view(np.uint64), x.view(np.uint64))
    order = np.argsort(k, kind="stable")
    assert np.all(np.diff(x[order]) >= 0)
    assert st.radix_keys(np.array([-0.0]))[0] + np.uint64(1) == st.radix_keys(np.array([0.0]))[0]


def test_population_is_that_of_the_moments():
    """The order statistics reduce the entries the moments reduce (K5: |x| <= 1.79e308), so the global counts taken
    from the moments are the selection's counts. The doubles above 1.79e308 fall outside, like NaN and +-inf."""
    col = adversarial_columns()["huge"]
    assert list(st.k5_finite(col)) == [True, True, False, False, True, True]
    assert list(st.k5_finite([np.nan, np.inf, -np.inf, 1.79e308, -1.79e308])) == [False, False, False, True, True]


@pytest.mark.parametrize("name", list(adversarial_columns()))
def test_radix_protocol_equals_np_quantile(name):
    col = adversarial_columns()[name]
    got = st.distributed_quantiles_protocol(col[None, :], QS)[:, 0]
    assert _same(got, _np_quantile(col, QS)), (name, got, _np_quantile(col, QS))


def test_integer_virtual_index_and_many_columns():
    """q whose (n - 1) q is an integer (then gamma = 0), more quantiles than one call's selector cap (16), and several
    columns of different finite counts in one table."""
    rng = np.random.default_rng(3)
    table = rng.normal(size=(5, 401))
    table[1, :200] = np.nan                        # 201 finite entries
    table[2, ::2] = np.inf
    qs = list(np.linspace(0.0, 1.0, 41))           # (400) q integral for every q; 41 > 16: three selection calls
    got = st.distributed_quantiles_protocol(table, qs)
    for c in range(5):
        assert _same(got[:, c], _np_quantile(table[c], qs)), c


def test_ranks_follow_numpy_indexes():
    import torch
    counts = torch.tensor([0.0, 1.0, 2.0, 10.0, 1001.0], dtype=torch.float64)
    qs = [0.0, 0.5, 1 / 3, 0.999999, 1.0]
    r = st.quantile_ranks(counts, qs).numpy().reshape(5, len(qs), 2)
    for c, n in enumerate(counts.numpy()):
        for i, q in enumerate(qs):
            v = (n - 1) * q
            lo = n - 1 if v >= n - 1 else np.floor(v)
            hi = n - 1 if v >= n - 1 else np.floor(v) + 1
            assert tuple(r[c, i]) == (max(lo, 0), max(hi, 0))


@pytest.mark.parametrize("bad", [[-0.1], [1.5], [np.nan], [np.inf], [], [[0.5]]])
def test_bad_quantiles_raise(bad):
    with pytest.raises(ValueError):
        st.check_quantiles(bad)


def test_argext_restatement_and_merge():
    table = np.array([[1.0, 3.0, 3.0, -2.0, -2.0, np.nan],
                      [np.nan, np.inf, -np.inf, np.nan, np.nan, np.nan],
                      [0.0, -0.0, 0.0, -0.0, 0.0, 0.0],
                      [5.0, np.inf, 5.0, -np.inf, 4.0, 5.0]])
    for base in (0, 1000):
        m = st.merge_argext(st.local_argext_numpy(table, base)[None])
        assert list(m["argmax"]) == [base + 1, -1, base + 0, base + 0]
        assert list(m["argmin"]) == [base + 3, -1, base + 0, base + 4]
        assert m["max"][1] == -np.inf and m["min"][1] == np.inf
    # shards merged in any cut equal the whole column (ties to the lowest global index)
    for cuts in ([0, 2, 6], [0, 1, 3, 6], [0, 0, 6], [0, 3, 3, 6]):
        parts = [st.local_argext_numpy(table[:, a:b], a) for a, b in zip(cuts, cuts[1:])]
        whole = st.merge_argext(st.local_argext_numpy(table)[None])
        merged = st.merge_argext(np.stack(parts))
        for k in whole:
            assert np.array_equal(merged[k], whole[k]), (cuts, k)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, table, qs, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        # uneven shards: rank r holds a different number of samples than shard_bounds would give
        cuts = np.linspace(0, table.shape[1], world + 1).astype(int)
        cuts[1] = max(cuts[1] - 37, 0)
        lo, hi = cuts[rank], cuts[rank + 1]
        qv = st.distributed_quantiles_protocol(table[:, lo:hi], qs)
        ax = st.distributed_argext_protocol(table[:, lo:hi])
        q.put((rank, qv, ax))
    finally:
        dist.destroy_process_group()


def _run(world, table, qs):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, table, qs, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = {r: (qv, ax) for r, qv, ax in (q.get(timeout=120) for _ in range(world))}
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return res


@pytest.mark.parametrize("world", [2, 3])
def test_gloo_sharded_quantiles_and_argext_equal_single_shard(world):
    cols = adversarial_columns()
    rng = np.random.default_rng(7)
    table = np.stack([rng.normal(size=600), rng.integers(0, 4, size=600).astype(np.float64),
                      np.resize(cols["mixed_nonfinite"], 600), np.full(600, np.nan),
                      np.resize(cols["subnormals"], 600)])
    single = st.distributed_quantiles_protocol(table, QS)
    res = _run(world, table, QS)
    for r in range(world):
        qv, ax = res[r]
        assert np.array_equal(qv.view(np.int64), single.view(np.int64)), r      # bit for bit
        for c in range(table.shape[0]):
            assert _same(qv[:, c], _np_quantile(table[c], QS)), (r, c)
            fin = np.flatnonzero(st.k5_finite(table[c]))
            if fin.size:
                v = table[c][fin]
                assert ax["argmax"][c] == fin[np.argmax(v)] and ax["argmin"][c] == fin[np.argmin(v)], (r, c)
                assert ax["max"][c] == v.max() and ax["min"][c] == v.min()
            else:
                assert ax["argmax"][c] == -1 and ax["argmin"][c] == -1
