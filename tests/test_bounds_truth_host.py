"""CPU tier of tests/test_bounds_truth.py: the K3 headers compiled with g++ (tests/hostmath: api.bounds for the
single-horizon form, range.cpp for the horizon range) against the 50-digit truth of tests/mp_truth.py — Gram extremes
on hard plants, the whole bound chain on cfg-sweep-f's own inputs, and the flags on both sides of every edge. The
same checks as the GPU file, on fewer samples, so that a regression in the formulas shows without a GPU."""
import numpy as np
import pytest

from oracle import np_sampler
from tests import bounds_truth_cases as bc
from tests import mp_truth as mt
from tests import test_horizon_range_host as hr
from tests.hostmath import api

pytestmark = pytest.mark.slow


def _host_single(A, B, Q, R, lo, hi, dA, dB, N, e, MV, x, strict, K=None):
    S = dA.shape[1]
    vec = lambda v: np.full(S, float(v)) if np.isscalar(v) else np.asarray(v, dtype=float)   # noqa: E731
    xs = np.repeat(np.asarray(x, dtype=float).reshape(-1, 1), S, axis=1) if np.size(x) == B.shape[0] else x
    Kin = None if K is None else np.repeat(np.asarray(K, dtype=float).reshape(-1, 1), S, axis=1)
    return api.bounds(A, B, Q, R, lo, hi, dA, dB, N, vec(e), vec(e), vec(MV), xs, Kin, bc.P3, 0.3, strict=strict)


def test_gram_extremes_hard_plants_host():
    """Matrix-free lambda_min(H^) and ||Gamma||^2 (single horizon and horizon range N = 1..N_max) within 1e-11 of the
    50-digit eigenvalues of the assembled matrices, on the plants of bounds_truth_cases.gram_plants; the dense route on
    the same inputs (LQMPC_K3_DENSE's A/B switch) within its backward-error bound."""
    jobs, meta = [], []
    for name, A, B, Q, R, Ns in bc.gram_plants():
        n, m = B.shape
        dA, dB = bc.gram_perturbations(name, n, m, S=1)
        scalar = np.allclose(Q, Q[0, 0] * np.eye(n)) and np.allclose(R, R[0, 0] * np.eye(m))
        for N in Ns:
            Ah, Bh = bc.model(A, B, dA, dB, 0)
            jobs.append((Ah, Bh, Q, R, N, False))
            meta.append((name, A, B, Q, R, dA, dB, N, scalar))
    truths = bc.pmap(bc.gram_truth_float, jobs)
    worst = {"single": 0.0, "range": 0.0, "dense": 0.0}
    ranges = {}
    for (name, A, B, Q, R, dA, dB, N, scalar), t in zip(meta, truths):
        n, m = B.shape
        lo, hi = -0.3 * np.ones(m), 0.3 * np.ones(m)
        g = _host_single(A, B, Q, R, lo, hi, dA, dB, N, 5e-3, 1.0, np.ones(n) * 0.1, strict=0)
        worst["single"] = max(worst["single"], *bc.assert_gram(g["min_H"][0], g["norm_Gamma"][0], t,
                                                               what=(name, N, "single")))
        key = name
        if key not in ranges:
            Nmax = max(Ns for nm, _, _, _, _, Ns in bc.gram_plants() if nm == name)
            ranges[key] = hr.bounds(1, A, B, Q, R, lo, hi, dA, dB, 1, max(Nmax), np.full(1, 5e-3), np.ones((max(Nmax), 1)),
                                    np.ones((n, 1)) * 0.1, bc.P3, 0.3)
        d = ranges[key]["detail"][N - 1]
        ih, ig = mt.BOUND_FIELDS.index("min_H"), mt.BOUND_FIELDS.index("norm_Gamma")
        worst["range"] = max(worst["range"], *bc.assert_gram(d[ih, 0], d[ig, 0], t, what=(name, N, "range")))
        if N * m <= 60 and scalar:
            gd = _host_single(A, B, Q, R, lo, hi, dA, dB, N, 5e-3, 1.0, np.ones(n) * 0.1, strict=3)
            tol = bc.dense_tol(N, m, t["cond_H"])
            e = bc.assert_gram(gd["min_H"][0], gd["norm_Gamma"][0], t, tol=tol, what=(name, N, "dense"))
            worst["dense"] = max(worst["dense"], max(e) / tol * 1e-9)
    print("largest relative error per route:", worst)


def test_dense_route_literal_kron_host():
    """The dense route with non-scalar weights in the literal kron ordering, up to (2, 1), rho 1.3, N = 50
    (cond(H^) ~ 1e11), within bounds_truth_cases.dense_tol."""
    rng = np.random.default_rng(31)
    cases = []
    for n, m, rho, N in ((2, 1, 1.3, 50), (2, 2, 1.4, 30), (2, 1, 1.117, 25), (3, 2, 0.9, 12)):
        A = bc._scaled(rng, n, rho)
        B = rng.normal(size=(n, m))
        Mq, Mr = rng.normal(size=(n, n)), rng.normal(size=(m, m))
        Q, R = Mq @ Mq.T + 0.5 * np.eye(n), Mr @ Mr.T + 0.5 * np.eye(m)
        cases.append((A, B, Q, R, N))
    truths = bc.pmap(bc.gram_truth_float, [(A, B, Q, R, N, True) for A, B, Q, R, N in cases])
    for (A, B, Q, R, N), t in zip(cases, truths):
        n, m = B.shape
        z = np.zeros((n * n, 1)), np.zeros((n * m, 1))
        g = _host_single(A, B, Q, R, -np.ones(m), np.ones(m), *z, N, 5e-3, 1.0, np.ones(n) * 0.1, strict=1)
        tol = bc.dense_tol(N, m, t["cond_H"])
        e = abs(g["min_H"][0] - t["min_H"]) / t["min_H"]
        print("dense literal kron n=%d m=%d N=%d cond(H^)=%.1e: min_H rel. err %.1e (tol %.1e)"
              % (n, m, N, t["cond_H"], e, tol))
        assert e <= tol
        assert abs(g["norm_Gamma"][0] ** 2 - t["cmax"]) / t["cmax"] <= bc.dense_tol(N, m, 1.0)


def _sweep_inputs(N_sys):
    gA, _, _ = np_sampler.sample_error_grid(20240522, 0, 2, 2, N_sys, bc.SWEEP_ERRORS, N_sys // 5, "f")
    gB, _, _ = np_sampler.sample_error_grid(20240522, 1, 2, 1, N_sys, bc.SWEEP_ERRORS, N_sys // 5, "f")
    dA = np.ascontiguousarray(gA.reshape(4, -1))           # s = j * n_err + i
    dB = np.ascontiguousarray(gB.reshape(2, -1))
    e = np.tile(bc.SWEEP_ERRORS, N_sys)
    return dA, dB, e


def test_bound_chain_sweep_inputs_host(known):
    """cfg-sweep-f's plant, box and seeded grids at every level, M_V from the ring solves, N in {1, 7, 25, 50}:
    samples chosen at the edges plus random ones, every field of the single-horizon and the range form against
    k3_truth within 1e-9 (1 + kappa), Gram extremes within 1e-11, N_0 / N_min equal away from ceil jumps, flags
    both ways."""
    A, B, Q, R, lo, hi = bc.SWEEP_A, bc.SWEEP_B, bc.SWEEP_Q, bc.SWEEP_R, bc.SWEEP_LO, bc.SWEEP_HI
    ring = np.array(known["single"]["x0_vec"])
    x = ring[:, 1]
    dA, dB, e = _sweep_inputs(20)
    S = dA.shape[1]
    mv = hr.mpc(1, A, B, Q, R, lo, hi, dA, dB, 1, 50, pts=ring.T)["M_V"]
    rng_form = hr.bounds(1, A, B, Q, R, lo, hi, dA, dB, 1, 50, e, mv, np.repeat(x[:, None], S, axis=1), bc.P3, 0.3)
    rng = np.random.default_rng(4)
    jobs, meta = [], []
    for N, n_edge, n_rand in ((1, 4, 20), (7, 4, 20), (25, 3, 12), (50, 2, 6)):
        single = _host_single(A, B, Q, R, lo, hi, dA, dB, N, e, mv[N - 1], x, strict=1)
        picks = bc.pick_decisive(single, rng, n_edge, n_rand)
        for s in picks:
            Ah, Bh = bc.model(A, B, dA, dB, s)
            jobs.append((Ah, Bh, Q, R, lo, hi, N, e[s], mv[N - 1, s], x, 0.3))
            meta.append((N, s, {k: single[k][s] for k in mt.BOUND_FIELDS}, int(single["flags"][s]),
                         {k: rng_form["detail"][N - 1, i, s] for i, k in enumerate(mt.BOUND_FIELDS)},
                         int(rng_form["flags"][N - 1, s])))
    truths = bc.pmap(bc.truth_sample, jobs)
    worst, skipped = {}, 0
    for (N, s, got, fl, gotr, flr), t in zip(meta, truths):
        for g in (got, gotr):
            errs, sk = bc.compare_fields(g, t)
            skipped += sk
            for k, v in errs.items():
                worst[k] = max(worst.get(k, 0.0), v)
    edge = bc.check_flags([m_[3] for m_ in meta] + [m_[5] for m_ in meta], truths + truths)
    print("samples %d, ceil-edge %d, flag-edge %d; largest error / (1 + kappa): %s"
          % (len(meta), skipped, edge, {k: "%.1e" % v for k, v in sorted(worst.items())}))
    assert skipped <= 2 and edge <= 2


def test_flags_both_sides_of_every_edge_host():
    """bounds_truth_cases.edge_cases through the single-horizon form (explicit gains where the edge needs one) and, for
    the DARE-gain samples, the range form: bit 32 iff the truth's 1 - xi - eta <= 0, bit 512 iff a log / sqrt argument
    is out of domain, except within the stated margin; few samples there."""
    A, B, Q, R, lo, hi = bc.SWEEP_A, bc.SWEEP_B, bc.SWEEP_Q, bc.SWEEP_R, bc.SWEEP_LO, bc.SWEEP_HI
    x = np.array([0.15, 0.1])
    cases = bc.edge_cases()
    truths = bc.pmap(bc.truth_sample, [(A + dA.reshape(2, 2), B + dB.reshape(2, 1), Q, R, lo, hi, N, e_, MV, x, 0.3,
                                        True, K, False) for _, dA, dB, N, e_, MV, K in cases])
    flags, tags = [], []
    for (tag, dA, dB, N, e_, MV, K), t in zip(cases, truths):
        g = _host_single(A, B, Q, R, lo, hi, dA.reshape(4, 1), dB.reshape(2, 1), N, e_, MV, x, 1, K=K)
        flags.append(int(g["flags"][0]))
        tags.append(tag)
        if K is None:
            r = hr.bounds(1, A, B, Q, R, lo, hi, dA.reshape(4, 1), dB.reshape(2, 1), N, N, np.full(1, e_),
                          np.full((1, 1), MV), x.reshape(2, 1), bc.P3, 0.3)
            assert r["flags"][0, 0] == flags[-1], (tag, N)
        errs, _ = bc.compare_fields({k: g[k][0] for k in mt.BOUND_FIELDS}, t,
                                    fields=[f for f in mt.BOUND_FIELDS if f not in ("alpha", "beta", "bound", "E_u",
                                                                                    "E_psi_u", "theta_u", "theta_x_u",
                                                                                    "norm_Gamma", "min_H")])
    for tag in sorted(set(tags)):
        sides = {(t["b32"], t["b512"]) for t, tg in zip(truths, tags) if tg == tag}
        print(tag, sorted(sides, key=str))
    # every edge is exercised on both sides
    assert {t["b32"] for t, tg in zip(truths, tags) if tg == "den"} >= {True, False}
    assert {t["b512"] for t, tg in zip(truths, tags) if tg in ("rho_cl", "sqrt")} >= {True, False}
    edge = bc.check_flags(flags, truths)
    assert edge <= 12, edge


def test_rho_K_exactly_one_host():
    """rho(A^ + B^K) = 0.6 in float64, so rho_K = (rho_cl + 0.4)^2 is exactly 1: the reference divides by 1 - rho_K = 0
    and raises (ZeroDivisionError on Python floats; with numpy scalars gamma = inf and math.ceil / math.log of NaN raise
    ValueError). The kernel's gamma is inf and its log argument arg1 inf, so only the rho_gamma test (NaN) raises
    DOMAIN_ERROR (512) there; BOUND_INVALID (32) follows from the NaN xi."""
    from oracle import np_oracle as o
    A, B = np.diag([0.6, 0.3]), np.array([[1.0], [0.5]])
    Q, R, lo, hi = 2.0 * np.eye(2), np.eye(1), np.array([-0.1]), np.array([0.1])
    K = np.zeros((1, 2))
    with pytest.raises((ValueError, ZeroDivisionError)):
        o.energy_decreasing(A, B, Q, R, lo, hi, 5, 5e-3, 5e-3, K, 0.05)
    z = np.zeros((4, 1)), np.zeros((2, 1))
    g = _host_single(A, B, Q, R, lo, hi, *z, 5, 5e-3, 0.05, np.array([0.1, 0.1]), 1, K=K)
    assert g["rho_cl"][0] == 0.6 and g["rho_K"][0] == 1.0
    assert g["flags"][0] & 512 and g["flags"][0] & 32
