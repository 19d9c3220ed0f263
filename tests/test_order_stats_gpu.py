"""GPU tier — exact column quantiles and arg-extremes (K5 radix selection / argext): value-equal to np.quantile and
to the numpy restatement, deterministic, wired into the error x horizon sweep, and traceable back to the sample."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from lq_mpc_b200 import stats as _stats
from tests.conftest import ROOT
from tests.test_order_stats import QS, _np_quantile, _same, adversarial_columns

pytestmark = pytest.mark.gpu


def _check_quantiles(engine, table, qs=QS):
    from lq_mpc_b200 import stats
    got = stats.column_quantiles(engine, table, qs)
    host = table.cpu().numpy() if hasattr(table, "cpu") else np.atleast_2d(table)
    for c in range(host.shape[0]):
        assert _same(got[:, c], _np_quantile(host[c], qs)), (c, got[:, c], _np_quantile(host[c], qs))
    return got


@pytest.mark.parametrize("S", [0, 1, 2, 3, 1000, 1_000_003])
def test_quantiles_equal_numpy(engine, S):
    rng = np.random.default_rng(S)
    t = np.stack([rng.normal(size=S), rng.integers(0, 5, size=S).astype(np.float64),
                  np.exp(rng.normal(scale=30.0, size=S)) * np.sign(rng.normal(size=S))])
    if S:
        t[2, rng.integers(0, S, size=max(S // 50, 1))] = np.inf
        t[0, rng.integers(0, S, size=max(S // 70, 1))] = np.nan
    _check_quantiles(engine, t)


def test_adversarial_columns_and_many_quantiles(engine):
    qs = list(np.linspace(0, 1, 37)) + [1 / 3, 0.999999]       # 39 quantiles: three selection calls
    for name, col in adversarial_columns().items():
        _check_quantiles(engine, col[None, :].copy(), qs)


def test_strided_and_misaligned_tables(engine):
    """ld > S (a column slice of a wider buffer) and a column pointer that is not 16-byte aligned."""
    import torch
    rng = np.random.default_rng(5)
    buf = torch.from_numpy(rng.normal(size=(6, 10_001))).cuda()
    for view in (buf[:, :9_000], buf[:, 1:9_001], buf[1:, 3:4_000], buf[2:3, 1:]):
        got = _check_quantiles(engine, view)
        from lq_mpc_b200 import stats
        ax = stats.column_argext(engine, view, index_base=7)
        host = view.cpu().numpy()
        assert np.array_equal(ax["argmax"], 7 + host.argmax(axis=1)) and np.array_equal(ax["max"], host.max(axis=1))
        assert np.array_equal(ax["argmin"], 7 + host.argmin(axis=1)) and np.array_equal(ax["min"], host.min(axis=1))
        assert got.shape == (len(QS), view.shape[0])


def test_k1_table_with_unstable_loops(engine):
    from lq_mpc_b200 import sampling as sp, stats
    A, B, Q, R = sp.synth_problem(4, 2, seed=0)
    engine.set_problem(A, B, Q, R, Q, None, None, 30)
    dA, dB, x0 = sp.synth_samples_soa(4, 2, 200_003, seed=3, e=0.3)      # ~0.1 % unstable loops
    r = engine.eval_batch(dA, dB, x0, 9, 10, want=("J", "rho", "ratio"))
    tab = r["table"].cpu().numpy()
    assert np.isinf(tab[0]).any(), "expected unstable loops (J = +inf) in the table"
    _check_quantiles(engine, r["table"])
    ax = stats.column_argext(engine, r["table"])
    ref = stats.merge_argext(stats.local_argext_numpy(tab)[None])
    for k in ref:
        assert np.array_equal(ax[k], ref[k]), k


def test_deterministic_across_calls_and_cta_counts(engine):
    """The same column alone (many CTAs) and inside a 600-column table (one or two CTAs per column), twice each."""
    import torch
    from lq_mpc_b200 import stats
    rng = np.random.default_rng(8)
    col = rng.normal(size=300_001)
    col[::97] = np.nan
    wide = np.tile(col, (600, 1))
    a = stats.column_quantiles(engine, col[None, :], QS)
    b = stats.column_quantiles(engine, col[None, :], QS)
    w = stats.column_quantiles(engine, torch.from_numpy(wide).cuda(), QS)
    assert np.array_equal(a.view(np.int64), b.view(np.int64))
    assert np.array_equal(np.repeat(a, 600, axis=1).view(np.int64), w.view(np.int64))
    x1 = stats.column_argext(engine, col[None, :])
    xw = stats.column_argext(engine, torch.from_numpy(wide).cuda())
    for k in x1:
        assert np.all(xw[k] == x1[k][0]), k


def test_radix_kernels_match_numpy_restatement_pass_by_pass(engine):
    import torch
    from lq_mpc_b200 import stats
    rng = np.random.default_rng(4)
    t = np.stack([rng.normal(size=5001), rng.integers(-3, 3, size=5001).astype(np.float64),
                  np.resize([0.0, -0.0, 5e-324, np.nan, -np.inf, 1e308], 5001)])
    counts = torch.from_numpy(stats.k5_finite(t).sum(axis=1).astype(np.float64))
    rank_d = stats.quantile_ranks(counts.cuda(), QS)
    rank_h = stats.quantile_ranks(counts, QS).numpy()
    pre_d, pre_h = torch.zeros_like(rank_d), np.zeros(rank_h.shape, dtype=np.uint64)
    td = torch.from_numpy(t).cuda()
    for p in range(8):
        hd = engine.column_radix_histogram_raw(td, pre_d, p)
        hh = stats.radix_histogram_numpy(t, pre_h, p)
        assert np.array_equal(hd.cpu().numpy(), hh), p
        engine.column_radix_select_raw(hd, p, rank_d, pre_d)
        stats.radix_select_numpy(hh, p, rank_h, pre_h)
        assert np.array_equal(pre_d.cpu().numpy().view(np.uint64), pre_h), p
        assert np.array_equal(rank_d.cpu().numpy(), rank_h), p


def test_argext_ties_index_base_and_empty(engine):
    from lq_mpc_b200 import stats
    t = np.array([[1.0, 3.0, 3.0, -2.0, -2.0, np.nan] * 3,
                  [np.nan, np.inf, -np.inf, np.nan, np.nan, np.nan] * 3,
                  [0.0, -0.0, 0.0, -0.0, 0.0, 0.0] * 3])
    for base in (0, 12_345_678_901):
        ax = stats.column_argext(engine, t, index_base=base)
        ref = stats.merge_argext(stats.local_argext_numpy(t, base)[None])
        for k in ref:
            assert np.array_equal(ax[k], ref[k]), (base, k)
    empty = stats.column_argext(engine, np.zeros((2, 0)))
    assert list(empty["argmax"]) == [-1, -1] and np.all(empty["max"] == -np.inf) and np.all(empty["min"] == np.inf)
    assert np.all(np.isnan(stats.column_quantiles(engine, np.zeros((2, 0)), QS)))


def test_abi_rejects_bad_arguments(engine):
    import torch
    from lq_mpc_b200.engine import EngineError
    t = torch.zeros((2, 10), dtype=torch.float64, device="cuda")
    with pytest.raises(EngineError):
        engine.column_radix_histogram_raw(t, torch.zeros((2, 33), dtype=torch.int64, device="cuda"), 0)
    with pytest.raises(EngineError):
        engine.column_radix_histogram_raw(t, torch.zeros((2, 4), dtype=torch.int64, device="cuda"), 8)
    with pytest.raises(EngineError):
        engine.column_argext_raw(t, -1)
    with pytest.raises(ValueError):
        from lq_mpc_b200 import stats
        stats.column_quantiles(engine, t, [1.01])


# ---------------------------------------------------------------------------------------------------- the sweep
ERROR_VEC = np.linspace(1e-3, 1e-2, 10)
SWEEP_Q = (0.05, 0.5, 0.95)


def _example_problem(engine):
    A = np.array([[1, 0.7], [0.12, 0.4]]); B = np.array([[1], [1.2]])
    Q, F_u = 2 * np.eye(2), np.array([[10.0], [-10.0]])
    engine.set_problem(A, B, Q, np.eye(1), Q, [-0.1], [0.1], 30)
    return F_u, Q


def _check_sweep(plain, full):
    from lq_mpc_b200.sweep import QUANTITIES
    for k in plain:
        if k in ("seconds", "wall_seconds", "phase_seconds", "tables"):
            continue
        a, b = np.atleast_1d(np.asarray(plain[k])), np.atleast_1d(np.asarray(full[k]))
        assert a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8)), k
    tabs = full["tables"]                                  # [n_h][q][n_err][N_sys]
    for qi, q in enumerate(QUANTITIES):
        assert full[q + "_quantile"].shape == (len(SWEEP_Q),) + full[q + "_max"].shape
        for h in range(tabs.shape[0]):
            for i in range(tabs.shape[2]):
                col = tabs[h, qi, i]
                assert _same(full[q + "_quantile"][:, i, h], _np_quantile(col, SWEEP_Q)), (q, h, i)
                fin = np.flatnonzero(_stats.k5_finite(col))
                j_max, j_min = full[q + "_argmax"][i, h], full[q + "_argmin"][i, h]
                if fin.size:
                    assert col[j_max - full["j0"]] == full[q + "_max"][i, h] and col[j_min - full["j0"]] == full[q + "_min"][i, h]
                    assert j_max - full["j0"] == fin[np.argmax(col[fin])] and j_min - full["j0"] == fin[np.argmin(col[fin])]
                else:
                    assert j_max == -1 and j_min == -1


@pytest.mark.parametrize("fused", [False, True])
def test_sweep_order_statistics_device_grids(engine, fused):
    from lq_mpc_b200 import sampling as sp
    from lq_mpc_b200.sweep import QUANTITIES, error_horizon_sweep
    F_u, Q = _example_problem(engine)
    horizons = [2, 3, 5, 9]
    eA, eB = sp.device_error_grids(engine, 2, 1, ERROR_VEC, 200, "f", seed=20240522)
    kw = dict(fused_horizons=fused)
    plain = error_horizon_sweep(engine, eA, eB, ERROR_VEC, horizons, F_u, Q, **kw)
    full = error_horizon_sweep(engine, eA, eB, ERROR_VEC, horizons, F_u, Q, quantiles=SWEEP_Q, worst=True,
                               keep_tables=True, **kw)
    full["j0"] = 0
    _check_sweep(plain, full)
    assert np.array_equal(full["quantiles"], SWEEP_Q)
    # shards of the device grid (j_first = the shard's first perturbation) merge to the unsharded indices
    from lq_mpc_b200 import stats
    parts = []
    for k in (0, 1):
        lo, hi = stats.shard_bounds(1000, k, 2)
        sA, sB = sp.device_error_grids(engine, 2, 1, ERROR_VEC, 200, "f", seed=20240522, j_first=lo, N_sys=hi - lo)
        part = error_horizon_sweep(engine, sA, sB, ERROR_VEC, horizons, F_u, Q, quantiles=SWEEP_Q, worst=True,
                                   keep_tables=True, j_first=lo, **kw)
        part["j0"] = lo
        _check_sweep({}, part)
        parts.append(part)
    for q in QUANTITIES:
        for ext, better in (("max", np.greater), ("min", np.less)):
            a, b = parts
            pick_b = better(b[q + "_" + ext], a[q + "_" + ext]) | (a[q + "_arg" + ext] < 0)
            merged = np.where(pick_b & (b[q + "_arg" + ext] >= 0), b[q + "_arg" + ext], a[q + "_arg" + ext])
            assert np.array_equal(merged, full[q + "_arg" + ext]), (q, ext)


def test_sweep_order_statistics_golden_grids(engine, golden):
    from lq_mpc_b200.sweep import error_horizon_sweep
    F_u, Q = _example_problem(engine)
    gA, gB = golden["error_A_f"], golden["error_B_f"]
    for fused in (False, True):
        plain = error_horizon_sweep(engine, gA, gB, ERROR_VEC, [1, 4, 6], F_u, Q, fused_horizons=fused)
        full = error_horizon_sweep(engine, gA, gB, ERROR_VEC, [1, 4, 6], F_u, Q, fused_horizons=fused,
                                   quantiles=SWEEP_Q, worst=True, keep_tables=True)
        full["j0"] = 0
        _check_sweep(plain, full)
        for k in (0, 1):                                   # shard (k, 2): indices stay global
            part = error_horizon_sweep(engine, gA, gB, ERROR_VEC, [1, 4, 6], F_u, Q, fused_horizons=fused,
                                       shard=(k, 2), quantiles=SWEEP_Q, worst=True, keep_tables=True)
            from lq_mpc_b200 import stats
            part["j0"] = stats.shard_bounds(gA.shape[2], k, 2)[0]
            _check_sweep({}, part)


def test_worst_index_regenerates_the_sample(engine):
    """argmax of true_cost and bound -> sampling.perturbation_at -> the S = 1 re-run gives the column max bit for bit."""
    import torch
    from lq_mpc_b200 import sampling as sp
    from lq_mpc_b200.sweep import error_horizon_sweep
    from lq_mpc_b200.utils import circle_generator
    F_u, Q = _example_problem(engine)
    horizons = [3, 7]
    N_matrix, seed = 200, 20240522
    eA, eB = sp.device_error_grids(engine, 2, 1, ERROR_VEC, N_matrix, "f", seed=seed)
    res = error_horizon_sweep(engine, eA, eB, ERROR_VEC, horizons, F_u, Q, worst=True)
    ring = circle_generator(8, 1.5, res["epsilon_lqr"], Q).T.copy()
    x_start = res["x_start"]
    for h, N in enumerate(horizons):
        for i in (0, 4, 9):
            for q, key in (("true_cost", "J_T"), ("bound", "bound")):
                j = int(res[q + "_argmax"][i, h])
                dA, dB = sp.perturbation_at(engine, seed, 2, 1, ERROR_VEC, N_matrix, "f", j, i)
                a, b = dA.reshape(4, 1), dB.reshape(2, 1)
                if q == "true_cost":
                    v = engine.simulate_batch(a, b, N, 30, x0_shared=x_start, want=("J_T", "flags"))["J_T"]
                else:
                    mv = engine.mpc_solve_batch(a, b, N, pts=ring, want=("M_V", "flags"))["M_V"]
                    e = torch.full((1,), ERROR_VEC[i], dtype=torch.float64, device="cuda")
                    v = engine.bounds_batch(a, b, N, e, e, mv, x_start, (0.1, 1.0, 0.6), res["V_expert"],
                                            strict_reference=True)["bound"]
                got = float(v.reshape(-1)[0].item())
                assert np.float64(got).view(np.int64) == np.float64(res[q + "_max"][i, h]).view(np.int64), (q, N, i, j)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("world", [2, 4, 8])
def test_nccl_sharded_order_statistics_equal_single_gpu(world):
    import torch
    if not torch.cuda.is_available() or torch.cuda.device_count() < world:
        pytest.skip("needs %d CUDA devices" % world)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "multigpu_order_stats_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "MULTIGPU_ORDER_STATS_OK world=%d" % world in r.stdout
