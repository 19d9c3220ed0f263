"""K3 (bounds_kernel, the horizon-range kernel and the run-time-dimension warp route) against the 50-digit truth of
tests/mp_truth.py: Gram extremes on hard plants (matrix-free within 1e-11, the dense route within its backward-error
bound), every field of the bound chain on cfg-sweep-f's own inputs (1e-9 times the field's condition factor), the
flags on both sides of every classification edge, and the sweep's n_invalid counts. Shared inputs and checks:
tests/bounds_truth_cases.py; the CPU tier of the same checks: tests/test_bounds_truth_host.py."""
import numpy as np
import pytest

from tests import bounds_truth_cases as bc
from tests import mp_truth as mt

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gram_cases():
    """Every (plant, N, sample) of bounds_truth_cases.gram_plants with its 50-digit Gram extremes (time-major weights)."""
    jobs, meta = [], []
    for name, A, B, Q, R, Ns in bc.gram_plants():
        n, m = B.shape
        dA, dB = bc.gram_perturbations(name, n, m, S=2)
        for N in Ns:
            for s in range(2):
                Ah, Bh = bc.model(A, B, dA, dB, s)
                jobs.append((Ah, Bh, Q, R, N, False))
                meta.append((name, N, s))
    return dict(zip(meta, bc.pmap(bc.gram_truth_float, jobs)))


def _np(d):
    return {k: v.cpu().numpy() for k, v in d.items()}


def test_gram_extremes_hard_plants(engine, gram_cases, monkeypatch):
    """bounds_batch and bounds_range (N = 1..max listed N) hold lambda_min(H^) and ||Gamma||^2 to 1e-11 of the truth;
    LQMPC_K3_DENSE=1 (Gram matrix + Householder + Sturm) holds them to dense_tol."""
    monkeypatch.delenv("LQMPC_K3_DENSE", raising=False)
    worst = {"batch": 0.0, "range": 0.0, "dense": 0.0}
    for name, A, B, Q, R, Ns in bc.gram_plants():
        n, m = B.shape
        dA, dB = bc.gram_perturbations(name, n, m, S=2)
        engine.set_problem(A, B, Q, R, Q, -0.3 * np.ones(m), 0.3 * np.ones(m), 10)
        x = 0.1 * np.ones(n)
        scalar = np.allclose(Q, Q[0, 0] * np.eye(n)) and np.allclose(R, R[0, 0] * np.eye(m))
        rg = _np(engine.bounds_range(dA, dB, 1, max(Ns), 5e-3, 5e-3, 1.0, x, bc.P3, 0.3, strict_reference=False))
        for N in Ns:
            g = _np(engine.bounds_batch(dA, dB, N, 5e-3, 5e-3, 1.0, x, bc.P3, 0.3, strict_reference=False))
            for s in range(2):
                t = gram_cases[(name, N, s)]
                e = bc.assert_gram(g["min_H"][s], g["norm_Gamma"][s], t, what=(name, N, s, "batch"))
                worst["batch"] = max(worst["batch"], *e)
                e = bc.assert_gram(rg["min_H"][N - 1, s], rg["norm_Gamma"][N - 1, s], t, what=(name, N, s, "range"))
                worst["range"] = max(worst["range"], *e)
            if scalar and N * m <= 100:
                monkeypatch.setenv("LQMPC_K3_DENSE", "1")
                gd = _np(engine.bounds_batch(dA, dB, N, 5e-3, 5e-3, 1.0, x, bc.P3, 0.3))
                monkeypatch.delenv("LQMPC_K3_DENSE")
                for s in range(2):
                    t = gram_cases[(name, N, s)]
                    tol = bc.dense_tol(N, m, t["cond_H"])
                    e = bc.assert_gram(gd["min_H"][s], gd["norm_Gamma"][s], t, tol=tol, what=(name, N, s, "dense"))
                    worst["dense"] = max(worst["dense"], *e)
    print("largest relative error per route:", worst)


@pytest.mark.parametrize("n,m", [(5, 2), (12, 4)])
def test_gram_extremes_warp_route(engine, n, m):
    """The run-time-dimension route (one warp per sample) on unstable plants with scalar and non-scalar (time-major)
    weights: Gram extremes within 1e-11 of the truth."""
    rng = np.random.default_rng(50 + n)
    Ns = (1, 2, 12, 13, 30) if n == 5 else (1, 2, 12)
    cases = []
    for rho, general in ((1.117, False), (1.3, True)):
        A = bc._scaled(rng, n, rho)
        B = rng.normal(size=(n, m))
        if general:
            Uq, _ = np.linalg.qr(rng.normal(size=(n, n)))
            Q = Uq @ np.diag(np.logspace(0, 4, n)) @ Uq.T
            Mr = rng.normal(size=(m, m)); R = Mr @ Mr.T + np.eye(m)
        else:
            Q, R = 2.0 * np.eye(n), np.eye(m)
        cases.append((A, B, Q, R))
    jobs = [(A, B, Q, R, N, False) for A, B, Q, R in cases for N in Ns]
    truths = iter(bc.pmap(bc.gram_truth_float, jobs))
    worst = 0.0
    for A, B, Q, R in cases:
        engine.set_problem(A, B, Q, R, Q, -0.3 * np.ones(m), 0.3 * np.ones(m), 10)
        assert (n, m) not in engine.supported_dims()
        for N in Ns:
            g = _np(engine.bounds_batch(None, None, N, 1e-3, 1e-3, 1.0, 0.1 * np.ones(n), bc.P3, 0.3, S=1,
                                        strict_reference=False))
            worst = max(worst, *bc.assert_gram(g["min_H"][0], g["norm_Gamma"][0], next(truths), what=(n, m, N)))
    print("warp route (%d, %d): largest relative error %.1e" % (n, m, worst))


def test_dense_route_literal_kron(engine):
    """Non-scalar weights in the literal kron ordering take the dense route: within dense_tol of the truth up to
    (2, 1), rho 1.3, N = 50 (cond(H^) ~ 1e11)."""
    rng = np.random.default_rng(31)
    cases = []
    for n, m, rho, N in ((2, 1, 1.3, 50), (2, 2, 1.4, 30), (2, 1, 1.117, 25), (3, 2, 0.9, 12)):
        A = bc._scaled(rng, n, rho)
        B = rng.normal(size=(n, m))
        Mq, Mr = rng.normal(size=(n, n)), rng.normal(size=(m, m))
        cases.append((A, B, Mq @ Mq.T + 0.5 * np.eye(n), Mr @ Mr.T + 0.5 * np.eye(m), N))
    truths = bc.pmap(bc.gram_truth_float, [(A, B, Q, R, N, True) for A, B, Q, R, N in cases])
    for (A, B, Q, R, N), t in zip(cases, truths):
        n, m = B.shape
        engine.set_problem(A, B, Q, R, Q, -np.ones(m), np.ones(m), 10)
        g = _np(engine.bounds_batch(None, None, N, 5e-3, 5e-3, 1.0, 0.1 * np.ones(n), bc.P3, 0.3, S=1))
        tol = bc.dense_tol(N, m, t["cond_H"])
        e = abs(g["min_H"][0] - t["min_H"]) / t["min_H"]
        print("dense literal kron n=%d m=%d N=%d cond(H^)=%.1e: min_H rel. err %.1e (tol %.1e)"
              % (n, m, N, t["cond_H"], e, tol))
        assert e <= tol
        assert abs(g["norm_Gamma"][0] ** 2 - t["cmax"]) / t["cmax"] <= bc.dense_tol(N, m, 1.0)


@pytest.fixture(scope="module")
def sweep_setup(engine):
    """cfg-sweep-f's problem on the engine, 200 perturbations per level from the seeded device grids, x_start,
    V_expert and the ring M_V of every horizon 1..50."""
    from lq_mpc_b200 import sampling as sp
    from lq_mpc_b200.utils import circle_generator, local_radius
    A, B, Q, R, lo, hi = bc.SWEEP_A, bc.SWEEP_B, bc.SWEEP_Q, bc.SWEEP_R, bc.SWEEP_LO, bc.SWEEP_HI
    engine.set_problem(A, B, Q, R, Q, lo, hi, 30)
    dA, dB = sp.device_error_grids(engine, 2, 1, bc.SWEEP_ERRORS, 40, "f", seed=20240522)
    F_u = np.array([[10.0], [-10.0]])
    K_lqr = engine.dlqr_batch(S=1)["K"].cpu().numpy()[:, 0].reshape(-1, 2)
    ring = circle_generator(8, 1.5, local_radius(F_u, -K_lqr, Q), Q)
    x = ring[:, 1].copy()
    V_exp = float(engine.mpc_solve_batch(None, None, 30, pts=x[None], S=1)["V"][0, 0])
    mv = engine.mpc_solve_range(dA, dB, 1, 50, pts=engine._dev(ring.T.copy()), want=("M_V",))["M_V"]
    e = np.tile(bc.SWEEP_ERRORS, dA.shape[1] // len(bc.SWEEP_ERRORS))
    return dict(dA=dA, dB=dB, e=e, x=x, V_exp=V_exp, mv=mv, F_u=F_u)


def test_bound_chain_sweep_inputs(engine, sweep_setup):
    """Every field of bounds_batch and bounds_range on cfg-sweep-f's inputs (all levels, N in {1, 7, 25, 50}), on
    samples chosen at the edges plus random ones, against k3_truth: 1e-9 (1 + kappa), Gram extremes 1e-11; N_0 / N_min
    equal away from ceil jumps; flags both ways; range and single-horizon flags equal everywhere."""
    A, B, Q, R, lo, hi = bc.SWEEP_A, bc.SWEEP_B, bc.SWEEP_Q, bc.SWEEP_R, bc.SWEEP_LO, bc.SWEEP_HI
    st = sweep_setup
    dA, dB, e, x, V_exp, mv = (st[k] for k in ("dA", "dB", "e", "x", "V_exp", "mv"))
    ed = engine._dev(e)
    rg = _np(engine.bounds_range(dA, dB, 1, 50, ed, ed, mv, x, bc.P3, V_exp))
    dAn, dBn, mvn = dA.cpu().numpy(), dB.cpu().numpy(), mv.cpu().numpy()
    rng = np.random.default_rng(4)
    jobs, meta = [], []
    for N, n_edge, n_rand in ((1, 15, 120), (7, 15, 120), (25, 10, 60), (50, 8, 30)):
        g = _np(engine.bounds_batch(dA, dB, N, ed, ed, mv[N - 1], x, bc.P3, V_exp))
        assert np.array_equal(g["flags"], rg["flags"][N - 1])
        for s in bc.pick_decisive(g, rng, n_edge, n_rand):
            Ah, Bh = bc.model(A, B, dAn, dBn, s)
            jobs.append((Ah, Bh, Q, R, lo, hi, N, e[s], mvn[N - 1, s], x, V_exp))
            meta.append(({k: g[k][s] for k in mt.BOUND_FIELDS}, int(g["flags"][s]),
                         {k: rg[k][N - 1, s] for k in mt.BOUND_FIELDS}))
    truths = bc.pmap(bc.truth_sample, jobs)
    worst, skipped = {}, 0
    for (got, fl, gotr), t in zip(meta, truths):
        for gg in (got, gotr):
            errs, sk = bc.compare_fields(gg, t)
            skipped += sk
            for k, v in errs.items():
                worst[k] = max(worst.get(k, 0.0), v)
    edge = bc.check_flags([m_[1] for m_ in meta], truths)
    print("samples %d, ceil-edge %d, flag-edge %d; largest error / (1 + kappa): %s"
          % (len(meta), skipped, edge, {k: "%.1e" % v for k, v in sorted(worst.items())}))
    assert skipped <= 4 and edge <= 4


def test_flags_both_sides_of_every_edge(engine):
    """bounds_truth_cases.edge_cases through bounds_batch and bounds_range (N_min = N_max = N) with the same gain:
    bit 32 iff the truth's 1 - xi - eta <= 0, bit 512 iff a log / sqrt argument is out of domain, except within the
    stated margin; few samples there; range and single-horizon flags equal."""
    A, B, Q, R, lo, hi = bc.SWEEP_A, bc.SWEEP_B, bc.SWEEP_Q, bc.SWEEP_R, bc.SWEEP_LO, bc.SWEEP_HI
    engine.set_problem(A, B, Q, R, Q, lo, hi, 30)
    x = np.array([0.15, 0.1])
    cases = bc.edge_cases()
    truths = bc.pmap(bc.truth_sample, [(A + dA.reshape(2, 2), B + dB.reshape(2, 1), Q, R, lo, hi, N, e_, MV, x, 0.3,
                                        True, K, False) for _, dA, dB, N, e_, MV, K in cases])
    flags = []
    for (tag, dA, dB, N, e_, MV, K), t in zip(cases, truths):
        args = (dA.reshape(4, 1), dB.reshape(2, 1))
        g = _np(engine.bounds_batch(*args, N, e_, e_, MV, x, bc.P3, 0.3, K=K, S=1))
        r = _np(engine.bounds_range(*args, N, N, e_, e_, MV, x, bc.P3, 0.3, K=K, S=1))
        assert int(r["flags"][0, 0]) == int(g["flags"][0]), (tag, N)
        flags.append(int(g["flags"][0]))
        bc.compare_fields({k: g[k][0] for k in mt.BOUND_FIELDS}, t,
                          fields=[f for f in mt.BOUND_FIELDS if f not in ("alpha", "beta", "bound", "E_u", "E_psi_u",
                                                                          "theta_u", "theta_x_u", "norm_Gamma",
                                                                          "min_H")])
    edge = bc.check_flags(flags, truths)
    assert edge <= 12, edge


@pytest.mark.parametrize("fused", [False, True])
def test_sweep_invalid_counts(engine, sweep_setup, fused):
    """error_horizon_sweep on 10 levels x N in {1, 7, 25, 50} x 200 perturbations: n_invalid of every cell equals the
    50-digit count of samples that are void (1 - xi - eta <= 0) or raise in the reference, up to the listed edge
    samples; n_failed is 0."""
    from lq_mpc_b200.sweep import error_horizon_sweep
    A, B, Q, R, lo, hi = bc.SWEEP_A, bc.SWEEP_B, bc.SWEEP_Q, bc.SWEEP_R, bc.SWEEP_LO, bc.SWEEP_HI
    st = sweep_setup
    horizons = [1, 7, 25, 50]
    res = error_horizon_sweep(engine, st["dA"], st["dB"], bc.SWEEP_ERRORS, horizons, st["F_u"], Q, keep_tables=True,
                              fused_horizons=fused)
    assert np.all(res["n_failed"] == 0)
    n_err = len(bc.SWEEP_ERRORS)
    dAn, dBn = st["dA"].cpu().numpy(), st["dB"].cpu().numpy()
    S = dAn.shape[1]
    mi = list(mt_q := ("true_cost", "bound", "alpha", "beta", "xi", "eta", "M_V")).index("M_V")
    jobs, where = [], []
    for h, N in enumerate(horizons):
        mvt = res["tables"][h, mi]                           # [n_err][N_sys]
        for s in range(S):
            j, i = divmod(s, n_err)
            Ah, Bh = bc.model(A, B, dAn, dBn, s)
            jobs.append((Ah, Bh, Q, R, lo, hi, N, bc.SWEEP_ERRORS[i], mvt[i, j], res["x_start"], res["V_expert"],
                         True, None, False))
            where.append((h, i))
    assert len(mt_q) == len(res["tables"][0])
    truths = bc.pmap(bc.truth_sample, jobs)
    lo_cnt = np.zeros((n_err, len(horizons)))
    hi_cnt = np.zeros((n_err, len(horizons)))
    edges = []
    for (h, i), t, job in zip(where, truths, jobs):
        void = (t["b32"], t["b512"])
        if None in void and not (True in void):
            edges.append((horizons[h], i))
            hi_cnt[i, h] += 1
        elif True in void:
            lo_cnt[i, h] += 1
            hi_cnt[i, h] += 1
    print("edge samples (N, level):", edges)
    assert len(edges) <= 4
    assert np.all(lo_cnt <= res["n_invalid"]) and np.all(res["n_invalid"] <= hi_cnt), (lo_cnt, res["n_invalid"])


def test_rho_K_exactly_one(engine):
    """rho(A^ + B^K) = 0.6 in float64, so rho_K is exactly 1 and the reference raises on 1 / (1 - rho_K): only the
    rho_gamma test of the kernel sees it (gamma = inf, arg1 = inf > 0, rho_gamma NaN) — bit 512 in both forms."""
    from oracle import np_oracle as o
    A, B = np.diag([0.6, 0.3]), np.array([[1.0], [0.5]])
    Q, R, lo, hi = 2.0 * np.eye(2), np.eye(1), np.array([-0.1]), np.array([0.1])
    K = np.zeros((1, 2))
    with pytest.raises((ValueError, ZeroDivisionError)):
        o.energy_decreasing(A, B, Q, R, lo, hi, 5, 5e-3, 5e-3, K, 0.05)
    engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
    x = np.array([0.1, 0.1])
    g = _np(engine.bounds_batch(None, None, 5, 5e-3, 5e-3, 0.05, x, bc.P3, 0.3, K=K, S=1))
    r = _np(engine.bounds_range(None, None, 5, 5, 5e-3, 5e-3, 0.05, x, bc.P3, 0.3, K=K, S=1))
    assert g["rho_cl"][0] == 0.6 and g["rho_K"][0] == 1.0
    assert g["flags"][0] & 512 and g["flags"][0] & 32 and r["flags"][0, 0] == g["flags"][0]
