"""GPU tier — the horizon-range entry points (lqmpc_mpc_solve_range, lqmpc_bounds_range; Engine.mpc_solve_range,
Engine.bounds_range) against one single-horizon call per N, and the fused-horizon sweep against the default sweep.

  * ring solves: bit for bit (V, u0, M_V, flags, NaN payloads included), ring points and per-sample states;
  * bounds: every field within 1e-9 of bounds_batch (the Gram-spectrum extremes come from a bisection that shares its
    probes across horizons; the other fields are the same formulas, which the compiler may contract into FMAs
    differently in the two kernels), the horizon-independent fields equal in every horizon slot, equal flags,
    bit-equal K_out / P_out;
  * every compiled pair, N_min > 1, N_min == N_max and N_max = 50; grid-stride launches of >= 4 samples per thread;
    every case without a fused kernel (run-time dimensions, polytope, references, dense K3 route) and K_in / K_shared;
  * the golden horizon table; error_horizon_sweep(fused_horizons=True) vs the default mode, also sharded.
"""
import numpy as np
import pytest

from tests.conftest import relerr

pytestmark = pytest.mark.gpu
TOL = 1e-9
ALL_DIMS = [(1, 1), (2, 1), (2, 2), (3, 1), (3, 2), (3, 3), (4, 1), (4, 2), (4, 4), (6, 2), (8, 2)]
P3 = np.array([0.1, 1, 0.6])
HORIZON_FREE = ['epsilon_K', 'norm_A', 'norm_B', 'norm_K', 'rho_cl', 'bar_u', 'bar_d_u', 'C_K', 'rho_K', 'gamma',
                'rho_gamma', 'h']
RANGES = [(4, 9), (7, 7), (1, 50)]


def _same_bits(a, b):
    import torch
    if a.dtype == torch.float64:
        a, b = a.view(torch.int64), b.view(torch.int64)
    return torch.equal(a, b)


def _plant(rng, n, m, general=False):
    A = rng.normal(size=(n, n)); A *= rng.uniform(0.8, 1.1) / np.max(np.abs(np.linalg.eigvals(A)))
    B = rng.normal(size=(n, m))
    if general:
        Mq, Mr = rng.normal(size=(n, n)), rng.normal(size=(m, m))
        Q, R = Mq @ Mq.T / n + 0.5 * np.eye(n), Mr @ Mr.T / m + 0.3 * np.eye(m)
    else:
        Q, R = rng.uniform(0.5, 3) * np.eye(n), rng.uniform(0.1, 2) * np.eye(m)
    lo, hi = -rng.uniform(0.05, 0.4, size=m), rng.uniform(0.05, 0.4, size=m)
    return A, B, Q, R, lo, hi


def _batch(n, m, S, seed, e=0.005):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    dA = (torch.rand((n * n, S), device="cuda", dtype=torch.float64, generator=g) - 0.5) * (2 * e)
    dB = (torch.rand((n * m, S), device="cuda", dtype=torch.float64, generator=g) - 0.5) * (2 * e)
    x0 = torch.randn((n, S), device="cuda", dtype=torch.float64, generator=g)
    x0 *= 10 ** (2 * torch.rand(S, device="cuda", dtype=torch.float64, generator=g) - 1.5)   # saturating and tiny
    return dA, dB, x0


def check_solve_range(engine, dA, dB, N_min, N_max, **kw):
    r = engine.mpc_solve_range(dA, dB, N_min, N_max, **kw)
    for h, N in enumerate(range(N_min, N_max + 1)):
        s = engine.mpc_solve_batch(dA, dB, N, **kw)
        for k in ("V", "u0", "M_V", "flags"):
            assert _same_bits(r[k][h], s[k]), (k, N)
    return r


def check_bounds_range(engine, dA, dB, N_min, N_max, e, MV, x, **kw):
    """MV: [H][S] tensor (per horizon) or a scalar."""
    from lq_mpc_b200.engine import BOUND_FIELDS
    r = engine.bounds_range(dA, dB, N_min, N_max, e, e, MV, x, P3, 0.37, want_K=True, want_P=True, **kw)
    for h, N in enumerate(range(N_min, N_max + 1)):
        mv = MV[h] if hasattr(MV, "ndim") and MV.ndim == 2 else MV
        s = engine.bounds_batch(dA, dB, N, e, e, mv, x, P3, 0.37, want_K=True, want_P=True, **kw)
        assert torch_equal(r["flags"][h], s["flags"]), N
        for f in BOUND_FIELDS:
            assert relerr(r[f][h].cpu().numpy(), s[f].cpu().numpy()) <= TOL, (f, N)
        for f in HORIZON_FREE:
            assert _same_bits(r[f][h], r[f][0]), (f, N)
        if h == 0:
            for k in ("K", "P"):
                if kw.get("K") is None or k == "K":
                    assert _same_bits(r[k], s[k]), k
    return r


def torch_equal(a, b):
    import torch
    return torch.equal(a, b)


@pytest.mark.parametrize("n,m", ALL_DIMS)
def test_ranges_every_compiled_pair(engine, n, m):
    import torch
    rng = np.random.default_rng(7000 + 10 * n + m)
    A, B, Q, R, lo, hi = _plant(rng, n, m)
    engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
    S = 1500
    dA, dB, x0 = _batch(n, m, S, seed=n * 10 + m)
    pts = x0[:, :4].t().contiguous()
    for N_min, N_max in RANGES:
        r = check_solve_range(engine, dA, dB, N_min, N_max, pts=pts, S=S)
        assert torch.equal(r["M_V"], r["V"].amax(1))
        check_solve_range(engine, dA, dB, N_min, N_max, x0=x0)
        e = torch.full((S,), 5e-3, dtype=torch.float64, device="cuda")
        check_bounds_range(engine, dA, dB, N_min, N_max, e, r["M_V"], x0)
    # non-scalar weights with time-major ordering: also the fused matrix-free route
    A, B, Q, R, lo, hi = _plant(rng, n, m, general=True)
    engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
    check_bounds_range(engine, dA, dB, 2, 12, 4e-3, 1.5, x0, strict_reference=False)


@pytest.mark.parametrize("n,m", [(2, 1), (4, 2)])
def test_ranges_grid_stride_launch(engine, n, m, monkeypatch):
    """Every launched thread strides over >= 4 samples (one wave of resident CTAs, batch sized from the device)."""
    import torch
    monkeypatch.setenv("LQMPC_K2_WAVES", "1")
    monkeypatch.setenv("LQMPC_K3_RANGE_WAVES", "1")
    pr = torch.cuda.get_device_properties(0)
    S = 4 * pr.multi_processor_count * pr.max_threads_per_multi_processor
    rng = np.random.default_rng(8000 + n)
    A, B, Q, R, lo, hi = _plant(rng, n, m)
    engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
    dA, dB, x0 = _batch(n, m, S, seed=99 + n)
    pts = x0[:, :3].t().contiguous()
    r = check_solve_range(engine, dA, dB, 20, 24, pts=pts, S=S)
    check_solve_range(engine, dA, dB, 21, 23, x0=x0)
    e = 10 ** (-4 + 2 * torch.rand(S, device="cuda", dtype=torch.float64))
    check_bounds_range(engine, dA, dB, 20, 24, e, r["M_V"], x0)


def test_fallback_routes(engine, monkeypatch):
    """No fused kernel: run-time dimensions (5, 2), an input polytope, references, the dense K3 route (forced and
    literal kron with non-scalar weights); and K_in / K_shared on the fused K3 route."""
    import torch
    rng = np.random.default_rng(9000)
    # run-time-dimension route
    A, B, Q, R, lo, hi = _plant(rng, 5, 2)
    engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
    S = 300
    dA, dB, x0 = _batch(5, 2, S, seed=5)
    r = check_solve_range(engine, dA, dB, 3, 8, pts=x0[:, :3].t().contiguous(), S=S)
    check_solve_range(engine, dA, dB, 6, 6, x0=x0)
    check_bounds_range(engine, dA, dB, 3, 8, 5e-3, r["M_V"], x0)
    # polytope, references, dense route, K_in / K_shared on a compiled pair
    A, B, Q, R, lo, hi = _plant(rng, 3, 2)
    engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
    dA, dB, x0 = _batch(3, 2, S, seed=6)
    F = np.array([[3.0, 1.0], [-2.0, 0.5], [0.5, -4.0], [-1.0, -1.0]])
    engine.set_input_polytope(F, bar_u=0.3, bar_d_u=1.1)
    r = check_solve_range(engine, dA, dB, 2, 9, x0=x0)
    check_bounds_range(engine, dA, dB, 2, 9, 5e-3, r["M_V"], x0)
    engine.set_input_polytope(None)
    with engine.references(rng.normal(size=(3, 12)) * 0.1, rng.normal(size=(2, 12)) * 0.05):
        check_solve_range(engine, dA, dB, 4, 12, x0=x0)
        check_solve_range(engine, dA, dB, 4, 12, pts=x0[:, :2].t().contiguous(), S=S)
    K = torch.randn((6, S), dtype=torch.float64, device="cuda") * 0.3
    check_bounds_range(engine, dA, dB, 2, 7, 5e-3, 1.2, x0, K=K)
    check_bounds_range(engine, dA, dB, 2, 7, 5e-3, 1.2, x0, K=K[:, 0].cpu().numpy())   # shared (m*n,)
    monkeypatch.setenv("LQMPC_K3_DENSE", "1")
    check_bounds_range(engine, dA, dB, 2, 7, 5e-3, 1.2, x0)
    monkeypatch.delenv("LQMPC_K3_DENSE")
    A, B, Q, R, lo, hi = _plant(rng, 3, 2, general=True)
    engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
    check_bounds_range(engine, dA, dB, 2, 7, 5e-3, 1.2, x0, strict_reference=True)


def test_bounds_range_golden_horizon_table(engine, golden, example, known):
    A, B, Q, R, lo, hi = (example[x] for x in ("A", "B", "Q", "R", "lo", "hi"))
    engine.set_problem(A, B, Q, R, Q, lo, hi, 30)
    ring = np.array(known["single"]["x0_vec"]); x_start = ring[:, 1]
    eA = np.ascontiguousarray(golden["error_A_f"][:, :, :, 4]).reshape(4, -1)
    eB = np.ascontiguousarray(golden["error_B_f"][:, :, :, 4]).reshape(2, -1)
    hz = [int(N) for N in golden["horizon"]]
    N_lo, N_hi = min(hz), max(hz)
    mv = engine.mpc_solve_range(eA, eB, N_lo, N_hi, pts=ring.T, want=("M_V",))["M_V"]
    S = eA.shape[1]
    e = np.full(S, 5e-3)
    b = engine.bounds_range(eA, eB, N_lo, N_hi, e, e, mv, x_start, example["p"], float(golden["V_expert"]))
    for col, N in enumerate(hz):
        for k, gk in (("alpha", "alpha_table_horizon"), ("beta", "beta_table_horizon"), ("xi", "xi_table_horizon"),
                      ("bound", "bound_table_horizon")):
            assert relerr(b[k][N - N_lo].cpu().numpy(), golden[gk][:, col]) < TOL, (k, N)


def _compare_sweeps(a, b):
    from lq_mpc_b200.sweep import QUANTITIES
    for q in QUANTITIES:
        for st in ("max", "min", "mean", "std"):
            k = q + "_" + st
            if q in ("M_V", "true_cost"):
                assert np.array_equal(a[k].view(np.int64), b[k].view(np.int64)), k
            else:
                assert relerr(a[k], b[k]) <= TOL, k
    assert np.array_equal(a["n_invalid"], b["n_invalid"])
    assert np.array_equal(a["n_failed"], b["n_failed"])
    assert set(a["phase_seconds"]) == set(b["phase_seconds"])
    assert set(a) == set(b)


def test_fused_sweep_matches_default(engine):
    from lq_mpc_b200 import sampling as sp
    from lq_mpc_b200.sweep import error_horizon_sweep
    from oracle import np_sampler
    A = np.array([[1, 0.7], [0.12, 0.4]]); B = np.array([[1], [1.2]])
    Q, R, F_u = 2 * np.eye(2), np.eye(1), np.array([[10.0], [-10.0]])
    engine.set_problem(A, B, Q, R, Q, [-0.1], [0.1], 30)
    error_vec = np.linspace(1e-3, 1e-2, 10)
    horizons = [2, 3, 5, 9, 17]
    eA, eB = sp.device_error_grids(engine, 2, 1, error_vec, 400, "f", seed=20240522)
    kw = dict(phase_times=True)
    d = error_horizon_sweep(engine, eA, eB, error_vec, horizons, F_u, Q, **kw)
    f = error_horizon_sweep(engine, eA, eB, error_vec, horizons, F_u, Q, fused_horizons=True, **kw)
    _compare_sweeps(d, f)
    # host grids sharded over two ranks' slices (shard = (k, 2))
    gA, _, _ = np_sampler.sample_error_grid(20240522, 0, 2, 2, 300, error_vec, 60, "f")
    gB, _, _ = np_sampler.sample_error_grid(20240522, 1, 2, 1, 300, error_vec, 60, "f")
    for k in (0, 1):
        d = error_horizon_sweep(engine, gA, gB, error_vec, [1, 4, 6], F_u, Q, shard=(k, 2), **kw)
        f = error_horizon_sweep(engine, gA, gB, error_vec, [1, 4, 6], F_u, Q, shard=(k, 2), fused_horizons=True, **kw)
        _compare_sweeps(d, f)


def test_bounds_range_rejects_wrong_lengths(engine):
    """Per-sample e_A / e_B / M_V of the wrong length are refused before anything reaches the kernel."""
    import torch
    rng = np.random.default_rng(9100)
    A, B, Q, R, lo, hi = _plant(rng, 2, 1)
    engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
    S = 64
    dA, dB, x0 = _batch(2, 1, S, seed=9)
    short = torch.full((S - 1,), 5e-3, dtype=torch.float64, device="cuda")
    for kw in (dict(e_A=short, e_B=5e-3, M_V=1.0), dict(e_A=5e-3, e_B=short, M_V=1.0),
               dict(e_A=5e-3, e_B=5e-3, M_V=torch.ones((2, S), dtype=torch.float64, device="cuda"))):
        with pytest.raises(ValueError):
            engine.bounds_range(dA, dB, 3, 5, kw["e_A"], kw["e_B"], kw["M_V"], x0, P3, 0.37)
