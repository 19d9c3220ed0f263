"""GPU tier — lqmpc_simulate_inf_batch (K2c: infinite-horizon cost of the input-constrained closed loop, certified by
an invariant ellipsoid) on the B200: every compiled (n, m) pair and the run-time-dimension route against the numpy
oracle and the CPU-tier harness (tests/test_simulate_inf_host.py), the identity with K2b's J_T, the unconstrained
case against K1, both routes against each other, grid-stride launches, the error paths and the shipped sweep's inputs."""
import numpy as np
import pytest

from oracle import np_oracle as o
from tests.test_simulate_inf_host import (COMPILED_DIMS, FLAG_TAIL_UNCERTIFIED, case, check_vs_oracle, host_inf,
                                          host_tail, model)

pytestmark = pytest.mark.gpu


def _np(d):
    return {k: v.cpu().numpy() for k, v in d.items()}


def _run(engine, c, T_max=1000, **kw):
    engine.set_problem(c["A"], c["B"], c["Q"], c["R"], c["Q"], c["lo"], c["hi"], 10)
    if c["F"] is not None:
        engine.set_input_polytope(c["F"])
    try:
        return _np(engine.simulate_inf_batch(c["dA"], c["dB"], c["N"], T_max, x0=c["x0"], **kw))
    finally:
        if c["F"] is not None:
            engine.set_input_polytope(None)


@pytest.mark.parametrize("n,m", COMPILED_DIMS)
def test_every_compiled_pair_vs_oracle_and_host(engine, n, m):
    polys = (False, True) if m >= 2 else (False,)
    for poly in polys:
        c = case(n, m, (200 if poly else 100) + 10 * n + m, S=4 if poly else 6, poly=poly)
        g = _run(engine, c)
        assert check_vs_oracle(c, g["J_inf"], g["T_cert"], g["flags"]) >= 2
        J, Tc, fl = host_inf(c["A"], c["B"], c["Q"], c["R"], c["lo"], c["hi"], c["dA"], c["dB"], c["N"], 1000,
                             c["x0"], c["F"])
        ok = Tc >= 0
        assert np.array_equal(ok, g["T_cert"] >= 0) and np.array_equal(np.isinf(J), np.isinf(g["J_inf"]))
        assert np.all(np.abs(g["J_inf"][ok] - J[ok]) <= 1e-10 * J[ok])
        assert np.all(np.abs(g["T_cert"][ok] - Tc[ok]) <= 1)


@pytest.mark.parametrize("n,m", [(5, 1), (5, 2), (7, 3), (16, 4), (32, 8)])
def test_runtime_dimension_route_vs_oracle(engine, n, m):
    c = case(n, m, 700 + 10 * n + m, S=3 if n >= 16 else 5)
    g = _run(engine, c)
    assert check_vs_oracle(c, g["J_inf"], g["T_cert"], g["flags"]) >= 2


@pytest.mark.parametrize("n,m", [(2, 1), (4, 2)])
def test_identity_with_simulate_batch(engine, n, m):
    """J_inf = J_T(T) + x_T'(S - Q) x_T for T >= tau, with K2b's J_T and X on the device."""
    c = case(n, m, 300 + 10 * n + m, S=6)
    g = _run(engine, c)
    T = int(g["T_cert"].max()) + 3
    sim = _np(engine.simulate_batch(c["dA"], c["dB"], c["N"], T, x0=c["x0"], want=("J_T", "X")))
    done = 0
    for s in np.flatnonzero(g["T_cert"] >= 0):
        S = host_tail(c["A"], c["B"], c["Q"], c["R"], c["lo"], c["hi"], *model(c, s), c["N"])[0]
        xT = sim["X"][T, :, s]
        assert abs(sim["J_T"][s] + xT @ (S - c["Q"]) @ xT - g["J_inf"][s]) <= 1e-9 * g["J_inf"][s]
        done += 1
    assert done >= 3


@pytest.mark.parametrize("n,m", [(2, 1), (3, 2), (4, 2), (8, 2), (5, 2)])
def test_no_bounds_matches_eval_batch(engine, n, m):
    import torch
    rng = np.random.default_rng(400 + n + m)
    A = rng.normal(size=(n, n)); A *= 0.9 / o.spectral_radius(A)
    B, Q, R = rng.normal(size=(n, m)), np.eye(n), 0.5 * np.eye(m)
    N, S = 6, 64
    dA = rng.uniform(-0.01, 0.01, size=(n * n, S)); dB = rng.uniform(-0.01, 0.01, size=(n * m, S))
    x0 = rng.normal(size=(n, S))
    engine.set_problem(A, B, Q, R, Q, None, None, 10)
    g = _np(engine.simulate_inf_batch(dA, dB, N, 0, x0=x0))
    T = lambda a: torch.as_tensor(a, dtype=torch.float64, device=engine.device)   # noqa: E731
    J = engine.eval_batch(T(dA), T(dB), T(x0), N, N, want=("J",))["J"][0].cpu().numpy()
    fin = np.isfinite(J)
    assert fin.sum() > S // 2
    assert np.array_equal(np.isinf(g["J_inf"]), ~fin)
    assert np.all(g["T_cert"][fin] == 0) and not np.any(g["flags"][fin])
    assert np.all(np.abs(g["J_inf"][fin] - J[fin]) <= 1e-12 * J[fin])


def test_compiled_and_runtime_routes_agree(engine, monkeypatch):
    c = case(4, 2, 801, S=32)
    a = _run(engine, c)
    monkeypatch.setenv("LQMPC_FORCE_DYN", "1")
    b = _run(engine, c)
    monkeypatch.delenv("LQMPC_FORCE_DYN")
    ok = a["T_cert"] >= 0
    assert ok.sum() >= 8 and np.array_equal(ok, b["T_cert"] >= 0)
    assert np.all(np.abs(a["J_inf"][ok] - b["J_inf"][ok]) <= 1e-12 * a["J_inf"][ok])
    # J_inf does not depend on tau: the certified step itself pins the run-time route's c_S (its own certificate and
    # LDL'-based lambda_max) against the compiled one
    assert np.array_equal(a["T_cert"], b["T_cert"]) and np.sum(a["T_cert"] >= 2) >= 4
    assert np.array_equal(a["flags"], b["flags"])


def test_grid_stride_launch_equals_gathered_sub_batches(engine):
    """A batch several waves of the capped grid deep (N >= 20: one wave of resident CTAs) is bit-equal, sample by
    sample, to sub-batches gathered from it."""
    rng = np.random.default_rng(901)
    c = case(2, 1, 902, S=1)
    S, N = 200_000, 20
    c["N"] = N
    c["dA"] = rng.uniform(-0.01, 0.01, size=(4, S)); c["dB"] = rng.uniform(-0.01, 0.01, size=(2, S))
    c["x0"] = np.repeat(c["x0"], S, axis=1) * rng.uniform(0.5, 1.5, size=S)
    full = _run(engine, c)
    assert np.sum(full["T_cert"] > 0) > S // 10
    for idx in (np.arange(0, S, 7), np.arange(S - 1000, S)):
        sub = dict(c, dA=c["dA"][:, idx].copy(), dB=c["dB"][:, idx].copy(), x0=c["x0"][:, idx].copy())
        g = _run(engine, sub)
        for k in ("J_inf", "T_cert", "flags"):
            assert np.array_equal(g[k], full[k][idx], equal_nan=(k == "J_inf")), k


def test_error_paths(engine):
    from lq_mpc_b200.engine import EngineError
    c = case(2, 1, 903, S=4)
    engine.set_problem(c["A"], c["B"], c["Q"], c["R"], c["Q"], c["lo"], c["hi"], 10)
    with engine.references(np.zeros((2, 20)) + 0.1, np.zeros((1, 20))):
        with pytest.raises(EngineError):
            engine.simulate_inf_batch(c["dA"], c["dB"], c["N"], 100, x0=c["x0"])
    with pytest.raises(EngineError):
        engine.simulate_inf_batch(c["dA"], c["dB"], c["N"], -1, x0=c["x0"])
    with pytest.raises(EngineError):
        engine.simulate_inf_batch(c["dA"], c["dB"], c["N"], 100, x0_shared=c["x0"][:, 0], x0=c["x0"])
    with pytest.raises(EngineError):
        engine.simulate_inf_batch(c["dA"], c["dB"], c["N"], 100)
    g = _np(engine.simulate_inf_batch(c["dA"], c["dB"], c["N"], 100, x0=c["x0"]))     # usable after the refusals
    assert np.all(g["T_cert"] >= 0) or np.any(g["flags"] & FLAG_TAIL_UNCERTIFIED)


def test_golden_inputs(engine, golden, example):
    z, ex = golden, example
    A, B, Q, R, lo, hi = ex["A"], ex["B"], ex["Q"], ex["R"], ex["lo"], ex["hi"]
    xs = o.circle_generator(8, 1.5, o.local_radius(lo, hi, -o.dlqr(A, B, Q, R)[0], Q), Q)[:, 1]
    eA, eB = z["error_A_f"], z["error_B_f"]
    engine.set_problem(A, B, Q, R, Q, lo, hi, 30)
    cells = [(i, 7, z["true_cost_error"][:, i]) for i in range(eA.shape[3])] + \
        [(4, int(N), z["true_cost_horizon"][:, h]) for h, N in enumerate(z["horizon"])]
    for i, N, col in cells:
        S = eA.shape[2]
        g = _np(engine.simulate_inf_batch(eA[:, :, :, i].reshape(4, S), eB[:, :, :, i].reshape(2, S), N, 1000,
                                          x0_shared=xs))
        assert np.all((g["T_cert"] >= 0) & (g["T_cert"] <= 30)) and not np.any(g["flags"] & ~2)
        assert np.max(np.abs(g["J_inf"] - col) / col) <= 1e-12


@pytest.mark.parametrize("fused", [False, True])
def test_sweep_infinite_horizon(engine, golden, fused):
    """error_horizon_sweep(infinite_horizon=True): every key of the plain sweep is bit-equal to a run without it, and on
    the shipped inputs (N = 7 over the error levels) true_cost_inf has the statistics of true_cost to 1e-12."""
    from lq_mpc_b200.sweep import QUANTITIES, error_horizon_sweep
    A = np.array([[1, 0.7], [0.12, 0.4]]); B = np.array([[1], [1.2]])
    Q, R, F_u = 2 * np.eye(2), np.eye(1), np.array([[10.0], [-10.0]])
    engine.set_problem(A, B, Q, R, Q, [-0.1], [0.1], 30)
    z = golden
    eA, eB = z["error_A_f"], z["error_B_f"]
    error_vec = np.linspace(1e-3, 1e-2, 10)
    kw = dict(fused_horizons=fused, quantiles=(0.1, 0.5, 0.9), worst=True)
    d = error_horizon_sweep(engine, eA, eB, error_vec, [7], F_u, Q, **kw)
    f = error_horizon_sweep(engine, eA, eB, error_vec, [7], F_u, Q, infinite_horizon=True, **kw)
    timing = {"seconds", "wall_seconds"}
    assert set(f) - set(d) == {"true_cost_inf_" + s for s in ("max", "min", "mean", "std", "quantile", "argmax",
                                                                 "argmin")} | {"ratio_true_inf_max", "n_uncertified",
                                                                               "n_inf"}
    for k in set(d) - timing:
        assert np.array_equal(np.asarray(d[k]), np.asarray(f[k])), k
    assert not np.any(f["n_uncertified"]) and not np.any(f["n_inf"])
    for s in ("max", "min", "mean"):
        assert np.max(np.abs(f["true_cost_inf_" + s] - f["true_cost_" + s]) / f["true_cost_" + s]) <= 1e-12, s
    assert np.max(np.abs(f["true_cost_inf_std"] - f["true_cost_std"]) / f["true_cost_std"]) <= 1e-9
    assert np.max(np.abs(f["true_cost_inf_quantile"] - f["true_cost_quantile"]) / f["true_cost_quantile"]) <= 1e-12
    assert np.max(np.abs(z["true_cost_error"].max(axis=0) - f["true_cost_inf_max"][:, 0]) /
                  z["true_cost_error"].max(axis=0)) <= 1e-12
    assert "true_cost_inf" not in QUANTITIES
