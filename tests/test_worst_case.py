"""GPU tier — lqmpc_eval_grad_batch / lqmpc_worst_case_batch (worst.cuh on the device, k_worst.cu) on the B200: the
device gradient against the CPU-tier harness (tests/test_worst_case_host.py) and the autograd oracle for every compiled
(n, m) pair, the value against K1, the ascent's checks and its agreement with the harness, grid-stride launches, batch
sizes, in-place outputs, the error paths and worst_case_search."""
import numpy as np
import pytest
import torch

from lq_mpc_b200.engine import FLAG_UNSTABLE, Engine, EngineError, _ptr
from tests.test_worst_case_host import (COMPILED_DIMS, N_OPC, ascent_cases, check_ascent, closed_loop_rho, feasible,
                                        host_ascent, host_grad, oracle_grad, plant, samples, synth)

pytestmark = pytest.mark.gpu


def _np(d):
    return {k: (v.cpu().numpy() if isinstance(v, torch.Tensor) else v) for k, v in d.items()}


def _set(engine, pb):
    A, B, Q, R, Pt = pb
    engine.set_problem(A, B, Q, R, Pt, None, None, N_OPC)


@pytest.mark.parametrize("n,m", COMPILED_DIMS)
def test_gradient_vs_harness_and_autograd(engine, n, m):
    rng = np.random.default_rng(500 + 10 * n + m)
    for N, scalar, general_P in ((1, True, False), (10, False, True), (30, True, True)):
        pb = plant(rng, n, m, rho=rng.uniform(0.85, 1.05), scalar=scalar, general_P=general_P)
        _set(engine, pb)
        dA, dB, x0 = samples(rng, n, m, 64, 0.02)
        g = _np(engine.eval_grad_batch(dA, dB, x0, N))
        h = host_grad(pb, dA, dB, x0, N)
        assert np.array_equal(g["flags"], h["flags"])
        ok = g["flags"] == 0
        assert ok.sum() >= 16          # N = 1 leaves many of these plants unstable
        for k in ("J", "ratio"):
            for s in np.flatnonzero(ok):
                assert abs(g[k][s] - h[k][s]) <= 1e-12 * abs(h[k][s])
        for k in ("gA", "gB"):
            for s in np.flatnonzero(ok):
                assert np.max(np.abs(g[k][:, s] - h[k][:, s])) <= 1e-12 * np.max(np.abs(h[k][:, s]))
        assert np.all(np.isnan(g["gA"][:, ~ok]))
        for s in np.flatnonzero(ok)[:3]:
            J, gA, gB = oracle_grad(pb, dA[:, s].reshape(n, n), dB[:, s].reshape(n, m), x0[:, s], N)
            ref = np.concatenate([gA.ravel(), gB.ravel()])
            got = np.concatenate([g["gA"][:, s], g["gB"][:, s]])
            assert np.max(np.abs(got - ref)) <= 1e-9 * np.max(np.abs(ref))
            assert abs(g["J"][s] - J) <= 1e-12 * abs(J)


@pytest.mark.parametrize("n,m", COMPILED_DIMS)
def test_value_matches_eval_batch(engine, n, m):
    rng = np.random.default_rng(600 + 10 * n + m)
    pb = plant(rng, n, m, rho=1.1)
    _set(engine, pb)
    dA, dB, x0 = samples(rng, n, m, 1000, 0.2)        # wide enough that some samples are unstable
    N = 6
    g = _np(engine.eval_grad_batch(dA, dB, x0, N))
    k1 = _np(engine.eval_batch(dA, dB, x0, N, N))
    assert np.array_equal(g["flags"], k1["flags"][0])
    assert np.max(np.abs(g["rho"] - k1["rho"][0])) <= 1e-14 * max(1.0, np.max(np.abs(k1["rho"][0])))
    fin = np.isfinite(k1["J"][0])
    assert np.array_equal(fin, np.isfinite(g["J"]))
    assert np.all(np.abs(g["J"][fin] - k1["J"][0][fin]) <= 1e-12 * np.abs(k1["J"][0][fin]))


@pytest.mark.parametrize("norm", ["max", "f", "2"])
def test_ascent_on_the_device(engine, norm):
    agree = total = conv = 0
    for pb, dA, dB, x0, N, eA, eB in ascent_cases():
        _set(engine, pb)
        got = _np(engine.worst_case_batch(dA, dB, x0, N, eA, eB, norm))
        start = _np(engine.worst_case_batch(dA, dB, x0, N, eA, eB, norm, max_iter=0))
        conv += check_ascent(pb, dA, dB, x0, N, eA, eB, norm, got, start["J"])
        # K1 at the returned perturbations reproduces J
        k1 = _np(engine.eval_batch(got["dA"], got["dB"], x0, N, N))
        fin = np.isfinite(got["J"])
        assert np.all(np.abs(k1["J"][0][fin] - got["J"][fin]) <= 1e-12 * got["J"][fin])
        h = host_ascent(pb, dA, dB, x0, N, eA, eB, norm)
        both = (got["flags"] == 0) & (h["flags"] == 0)
        total += both.sum()
        agree += np.sum(np.abs(got["J"][both] - h["J"][both]) <= 1e-9 * h["J"][both])
    assert conv >= 9 and total >= 6 and agree >= 0.99 * total


def test_ascent_destabilising_error_on_the_device(engine):
    A, B, Q, R = np.array([[1.3, 0.2], [0.0, 0.9]]), np.array([[1.0], [0.3]]), np.eye(2), np.eye(1)
    pb, N, e = (A, B, Q, R, Q), 8, 0.35
    _set(engine, pb)
    dA, dB, x0 = samples(np.random.default_rng(2), 2, 1, 8, 0.02)
    got = _np(engine.worst_case_batch(dA, dB, x0, N, e, e, "max"))
    hit = np.flatnonzero(got["flags"] & FLAG_UNSTABLE)
    assert len(hit) >= 1 and np.all(np.isinf(got["J"][hit]))
    for s in hit:
        assert closed_loop_rho(pb, got["dA"][:, s].reshape(2, 2), got["dB"][:, s].reshape(2, 1), N) >= 1 - 1e-12


def test_grid_stride_and_permutation(engine, monkeypatch):
    """Two CTAs of 128 threads for 2 000 samples (about 8 per thread): a permuted batch gives permuted results."""
    pb = synth()
    _set(engine, pb)
    rng = np.random.default_rng(9)
    dA, dB, x0 = samples(rng, 4, 2, 2000, 0.05)
    perm = rng.permutation(2000)
    monkeypatch.setenv("LQMPC_WORST_CTAS", "2")
    for call in (lambda a, b, x: engine.eval_grad_batch(a, b, x, 10),
                 lambda a, b, x: engine.worst_case_batch(a, b, x, 10, 0.05, 0.05, "f", max_iter=20)):
        r0 = _np(call(dA, dB, x0))
        r1 = _np(call(dA[:, perm], dB[:, perm], x0[:, perm]))
        for k, v in r0.items():
            assert np.array_equal(v[..., perm], r1[k], equal_nan=v.dtype.kind == "f"), k
    monkeypatch.delenv("LQMPC_WORST_CTAS")
    full = _np(engine.worst_case_batch(dA, dB, x0, 10, 0.05, 0.05, "f", max_iter=20))
    assert all(np.array_equal(full[k], r0[k], equal_nan=True) for k in r0)   # independent of the grid


@pytest.mark.parametrize("S", [1, 127, 129, 100003])
def test_batch_sizes(engine, S):
    pb = synth()
    _set(engine, pb)
    dA, dB, x0 = samples(np.random.default_rng(S), 4, 2, S, 0.01)
    g = _np(engine.eval_grad_batch(dA, dB, x0, 10))
    k1 = _np(engine.eval_batch(dA, dB, x0, 10, 10))
    assert np.all(np.abs(g["J"] - k1["J"][0]) <= 1e-12 * k1["J"][0])
    idx = np.unique(np.r_[0, S - 1, np.random.default_rng(1).integers(0, S, 8)])
    h = host_grad(pb, dA[:, idx], dB[:, idx], x0[:, idx], 10)
    assert np.max(np.abs(g["gA"][:, idx] - h["gA"])) <= 1e-12 * np.max(np.abs(h["gA"]))
    w = _np(engine.worst_case_batch(dA[:, :min(S, 2000)], dB[:, :min(S, 2000)], x0[:, :min(S, 2000)], 10, 0.01, 0.01,
                                    "max"))
    assert np.all(np.abs(w["dA"]) <= 0.01) and np.all(w["J"] >= k1["J"][0][:min(S, 2000)] * (1 - 1e-12))


def test_in_place_outputs_and_empty_batch(engine):
    pb = synth()
    _set(engine, pb)
    dA, dB, x0 = samples(np.random.default_rng(4), 4, 2, 300, 0.05)
    ref = _np(engine.worst_case_batch(dA, dB, x0, 10, 0.03, 0.03, "2"))
    tA, tB, tx = (torch.tensor(a, device=engine.device) for a in (dA, dB, x0))
    J = torch.empty(300, dtype=torch.float64, device=engine.device)
    rc = engine.lib.lqmpc_worst_case_batch(engine._h, 300, _ptr(tA), _ptr(tB), _ptr(tx), 10, 0.03, 0.03, 1, 200, 1e-8,
                                           _ptr(tA), _ptr(tB), _ptr(J), None, None, None, None)
    assert rc == 0
    engine.sync()
    assert np.array_equal(tA.cpu().numpy(), ref["dA"]) and np.array_equal(tB.cpu().numpy(), ref["dB"])
    assert np.array_equal(J.cpu().numpy(), ref["J"])
    n0 = engine.launch_count
    assert engine.lib.lqmpc_eval_grad_batch(engine._h, 0, None, None, None, 10, *[None] * 6) == 0
    assert engine.lib.lqmpc_worst_case_batch(engine._h, 0, None, None, None, 10, 0.1, 0.1, 0, 200, 1e-8,
                                             *[None] * 7) == 0
    assert engine.launch_count == n0


def test_error_paths(engine):
    EINVAL, ESTATE = -1, -4
    pb = synth()
    _set(engine, pb)
    dA, dB, x0 = (torch.zeros(k, 4, dtype=torch.float64, device=engine.device) for k in (16, 8, 4))
    p = [_ptr(dA), _ptr(dB), _ptr(x0)]

    def worst(N=10, eA=0.1, eB=0.1, norm=0, it=200, tol=1e-8, ctx=engine):
        return ctx.lib.lqmpc_worst_case_batch(ctx._h, 4, *p, N, eA, eB, norm, it, tol, *[None] * 7)

    assert engine.lib.lqmpc_eval_grad_batch(engine._h, 4, *p, 0, *[None] * 6) == EINVAL
    assert engine.lib.lqmpc_eval_grad_batch(engine._h, -1, *p, 10, *[None] * 6) == EINVAL
    assert engine.lib.lqmpc_eval_grad_batch(engine._h, 4, None, p[1], p[2], 10, *[None] * 6) == EINVAL
    for kw in (dict(N=0), dict(eA=-1e-3), dict(eB=float("inf")), dict(eA=float("nan")), dict(norm=3), dict(norm=-1),
               dict(it=-1), dict(tol=0.0), dict(tol=-1.0)):
        assert worst(**kw) == EINVAL, kw
    assert worst() == 0
    with pytest.raises(ValueError):
        engine.worst_case_batch(dA, dB, x0, 10, 0.1, 0.1, "fro")
    fresh = Engine(0)
    try:
        assert fresh.lib.lqmpc_eval_grad_batch(fresh._h, 4, *p, 10, *[None] * 6) == ESTATE
        assert worst(ctx=fresh) == ESTATE
        from lq_mpc_b200.sampling import synth_problem
        A4, B4, Q4, R4 = synth_problem(16, 4, seed=0)
        fresh.set_problem_tiled(A4, B4, Q4, R4, Q4, 12)
        assert fresh.lib.lqmpc_eval_grad_batch(fresh._h, 4, *p, 10, *[None] * 6) == EINVAL
        assert "tiled" in fresh.lib.lqmpc_last_error(fresh._h).decode()
        assert worst(ctx=fresh) == EINVAL
        A5, B5, Q5, R5 = synth_problem(5, 2, seed=0)
        fresh.set_problem(A5, B5, Q5, R5)
        assert fresh.lib.lqmpc_eval_grad_batch(fresh._h, 4, *p, 10, *[None] * 6) == EINVAL
        assert "run-time-dimension" in fresh.lib.lqmpc_last_error(fresh._h).decode()
        assert worst(ctx=fresh) == EINVAL
        with pytest.raises(EngineError):
            fresh.eval_grad_batch(np.zeros((25, 2)), np.zeros((10, 2)), np.zeros((5, 2)), 10)
    finally:
        fresh.close()


def test_worst_case_search(engine):
    from lq_mpc_b200.sampling import synth_problem, synth_samples_soa
    from lq_mpc_b200.worst_case import worst_case_search
    A, B, Q, R = synth_problem(4, 2, seed=0)
    engine.set_problem(A, B, Q, R, Q, None, None, 0)
    for norm, e in (("max", 0.05), ("f", 0.05)):
        if norm == "max":
            dA, dB, x0 = synth_samples_soa(4, 2, 3000, seed=1, e=e)
        else:
            from lq_mpc_b200.sampling import device_error_grids
            dA, dB = device_error_grids(engine, 4, 2, [e], 600, "f", allow_projected=True)
            x0 = np.random.default_rng(3).normal(size=4)
        r = worst_case_search(engine, dA, dB, x0, 10, e, e, norm, top_k=16)
        assert r["best_ratio"] >= r["sampled_max_ratio"]
        assert r["ratio_start"][0].item() == r["sampled_max_ratio"]
        gA, gB = r["dA"].cpu().numpy(), r["dB"].cpu().numpy()
        for s in range(gA.shape[1]):
            assert feasible(gA[:, s].reshape(4, 4), e, norm) and feasible(gB[:, s].reshape(4, 2), e, norm)
        assert np.all(r["ratio"].cpu().numpy() >= r["ratio_start"].cpu().numpy() * (1 - 1e-12))
