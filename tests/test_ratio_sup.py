"""GPU tier — lqmpc_ratio_sup_batch / lqmpc_worst_case_sup_batch (worst.cuh's SUP mode on the device, k_worst.cu) on
the B200: the worst ratio over every initial state gamma = lambda_max(S, P_exp), its worst state, eigengap and gradient
against the CPU-tier harness (tests/test_ratio_sup_host.py) for every compiled (n, m) pair, gamma against K1's ratio at
x0 = x_worst, the ascent's checks and its agreement with the harness, grid-stride launches, batch sizes, NULL and
in-place outputs, the error paths and worst_case_search_sup."""
import numpy as np
import pytest
import torch

from lq_mpc_b200.engine import FLAG_UNSTABLE, WORST_NORMS, Engine, EngineError, _ptr
from tests.test_ratio_sup_host import check_sup_ascent, host_sup, host_sup_ascent
from tests.test_worst_case_host import (COMPILED_DIMS, N_OPC, ascent_cases, closed_loop_rho, feasible, plant, samples,
                                        synth)

pytestmark = pytest.mark.gpu


def _np(d):
    return {k: (v.cpu().numpy() if isinstance(v, torch.Tensor) else v) for k, v in d.items()}


def _set(engine, pb):
    A, B, Q, R, Pt = pb
    engine.set_problem(A, B, Q, R, Pt, None, None, N_OPC)


@pytest.mark.parametrize("n,m", COMPILED_DIMS)
def test_ratio_sup_vs_harness(engine, n, m):
    rng = np.random.default_rng(900 + 10 * n + m)
    checked = 0
    for N, general in ((1, False), (10, True), (30, True)):
        pb = plant(rng, n, m, rho=rng.uniform(0.85, 1.05), scalar=not general, general_P=general)
        _set(engine, pb)
        dA, dB, _ = samples(rng, n, m, 64, 0.02)
        g = _np(engine.ratio_sup_batch(dA, dB, N, grad=True))
        v = _np(engine.ratio_sup_batch(dA, dB, N))
        h = host_sup(pb, dA, dB, N)
        for k in ("gamma", "gap", "x_worst", "rho", "flags"):
            assert np.array_equal(v[k], g[k], equal_nan=True), k     # the value-only call: the same value
        assert np.array_equal(g["flags"], h["flags"])
        ok = g["flags"] == 0                      # N = 1 leaves many of these plants unstable
        assert np.all(np.abs(g["gamma"][ok] - h["gamma"][ok]) <= 1e-12 * h["gamma"][ok])
        assert np.all(np.abs(g["gap"][ok] - h["gap"][ok]) <= 1e-12)
        assert np.all(np.isinf(g["gamma"][~ok])) and np.all(np.isnan(g["x_worst"][:, ~ok]))
        assert np.all(np.isnan(g["gap"][~ok])) and np.all(np.isnan(g["gA"][:, ~ok]))
        # x* and the gradient through it are determined to about eps / gap: a rounding difference in S moves the top
        # eigenvector by that much (a host build with FMA contraction differs from this harness by <= 1.1e-15 / gap)
        tol = np.maximum(1e-12, 2e-14 / h["gap"])
        for s in np.flatnonzero(ok):
            for k in ("x_worst", "gA", "gB"):
                d = np.max(np.abs(g[k][:, s] - h[k][:, s]))
                assert d <= tol[s] * np.max(np.abs(h[k][:, s])), (k, s, h["gap"][s])
        checked += ok.sum()
    assert checked >= 48


@pytest.mark.parametrize("n,m", COMPILED_DIMS)
def test_gamma_is_k1_ratio_at_x_worst(engine, n, m):
    rng = np.random.default_rng(1000 + 10 * n + m)
    pb = plant(rng, n, m, rho=1.3)
    _set(engine, pb)
    dA, dB, _ = samples(rng, n, m, 1000, 0.5)        # wide enough, and N short enough, that some samples are unstable
    N = 2
    g = _np(engine.ratio_sup_batch(dA, dB, N))
    k1 = _np(engine.eval_batch(dA, dB, np.where(np.isnan(g["x_worst"]), 1.0, g["x_worst"]), N, N))
    assert np.array_equal(g["flags"], k1["flags"][0])
    assert np.max(np.abs(g["rho"] - k1["rho"][0])) <= 1e-14 * max(1.0, np.max(np.abs(k1["rho"][0])))
    unstable = (g["flags"] & FLAG_UNSTABLE) != 0
    assert unstable.sum() >= 1 and (~unstable).sum() >= 20
    # gamma against K1's ratio on a moderate batch: next to rho = 1 K1's closed-form cost (n = 3, 4) and the doubling
    # here part by more than 1e-12
    rng = np.random.default_rng(1100 + 10 * n + m)
    pb = plant(rng, n, m, rho=1.1)
    _set(engine, pb)
    dA, dB, _ = samples(rng, n, m, 1000, 0.02)
    g = _np(engine.ratio_sup_batch(dA, dB, 6))
    k1 = _np(engine.eval_batch(dA, dB, np.where(np.isnan(g["x_worst"]), 1.0, g["x_worst"]), 6, 6))
    assert np.array_equal(g["flags"], k1["flags"][0])
    fin = (g["flags"] == 0) & (g["rho"] < 0.99)
    assert fin.sum() >= 800
    assert np.all(np.abs(k1["ratio"][0][fin] - g["gamma"][fin]) <= 1e-12 * g["gamma"][fin])


@pytest.mark.parametrize("norm", ["max", "f", "2"])
def test_ascent_on_the_device(engine, norm):
    agree = total = conv = 0
    for pb, dA, dB, _, N, eA, eB in ascent_cases():
        _set(engine, pb)
        got = _np(engine.worst_case_sup_batch(dA, dB, N, eA, eB, norm))
        start = _np(engine.worst_case_sup_batch(dA, dB, N, eA, eB, norm, max_iter=0))
        conv += check_sup_ascent(pb, dA, dB, N, eA, eB, norm, got, start["gamma"])
        fin = np.isfinite(got["gamma"])
        k1 = _np(engine.eval_batch(got["dA"], got["dB"], np.where(fin, got["x_worst"], 1.0), N, N))
        assert np.all(np.abs(k1["ratio"][0][fin] - got["gamma"][fin]) <= 1e-12 * got["gamma"][fin])
        h = host_sup_ascent(pb, dA, dB, N, eA, eB, norm)
        both = (got["flags"] == 0) & (h["flags"] == 0)
        total += both.sum()
        agree += np.sum(np.abs(got["gamma"][both] - h["gamma"][both]) <= 1e-9 * h["gamma"][both])
    assert conv >= 4 and total >= 4 and agree >= 0.99 * total


def test_ascent_destabilising_error_on_the_device(engine):
    A, B, Q, R = np.array([[1.3, 0.2], [0.0, 0.9]]), np.array([[1.0], [0.3]]), np.eye(2), np.eye(1)
    pb, N, e = (A, B, Q, R, Q), 8, 0.35
    _set(engine, pb)
    dA, dB, _ = samples(np.random.default_rng(2), 2, 1, 8, 0.02)
    got = _np(engine.worst_case_sup_batch(dA, dB, N, e, e, "max"))
    hit = np.flatnonzero(got["flags"] & FLAG_UNSTABLE)
    assert len(hit) >= 1 and np.all(np.isinf(got["gamma"][hit])) and np.all(np.isnan(got["x_worst"][:, hit]))
    for s in hit:
        assert closed_loop_rho(pb, got["dA"][:, s].reshape(2, 2), got["dB"][:, s].reshape(2, 1), N) >= 1 - 1e-12


def test_grid_stride_and_permutation(engine, monkeypatch):
    """Two CTAs of 128 threads for 2 000 samples (about 8 per thread): a permuted batch gives permuted results, and
    the same bits as one sample per thread."""
    pb = synth()
    _set(engine, pb)
    rng = np.random.default_rng(9)
    dA, dB, _ = samples(rng, 4, 2, 2000, 0.05)
    perm = rng.permutation(2000)
    calls = (lambda a, b: engine.ratio_sup_batch(a, b, 10, grad=True),
             lambda a, b: engine.ratio_sup_batch(a, b, 10),
             lambda a, b: engine.worst_case_sup_batch(a, b, 10, 0.05, 0.05, "f", max_iter=20))
    monkeypatch.setenv("LQMPC_WORST_CTAS", "2")
    strided = []
    for call in calls:
        r0 = _np(call(dA, dB))
        r1 = _np(call(dA[:, perm], dB[:, perm]))
        for k, v in r0.items():
            assert np.array_equal(v[..., perm], r1[k], equal_nan=v.dtype.kind == "f"), k
        strided.append(r0)
    monkeypatch.delenv("LQMPC_WORST_CTAS")
    for call, r0 in zip(calls, strided):
        full = _np(call(dA, dB))
        assert all(np.array_equal(full[k], r0[k], equal_nan=True) for k in r0)


@pytest.mark.parametrize("S", [1, 127, 129])
def test_batch_sizes(engine, S):
    pb = synth()
    _set(engine, pb)
    dA, dB, _ = samples(np.random.default_rng(S), 4, 2, S, 0.01)
    g = _np(engine.ratio_sup_batch(dA, dB, 10, grad=True))
    h = host_sup(pb, dA, dB, 10)
    assert np.array_equal(g["flags"], h["flags"]) and np.all(g["flags"] == 0)
    assert np.all(np.abs(g["gamma"] - h["gamma"]) <= 1e-12 * h["gamma"])
    # the synthetic plant's top eigenvalues lie 1e-5..1e-4 apart (relative): x* and the gradient are exact to eps / gap
    tol = np.maximum(1e-12, 1e-14 / h["gap"])
    for k in ("x_worst", "gA", "gB"):
        assert np.all(np.max(np.abs(g[k] - h[k]), axis=0) <= tol * np.max(np.abs(h[k]), axis=0)), k
    w = _np(engine.worst_case_sup_batch(dA, dB, 10, 0.01, 0.01, "max"))
    assert np.all(np.abs(w["dA"]) <= 0.01) and np.all(w["gamma"] >= g["gamma"] * (1 - 1e-12))


def test_null_and_in_place_outputs_and_empty_batch(engine):
    pb = synth()
    _set(engine, pb)
    dA, dB, _ = samples(np.random.default_rng(4), 4, 2, 300, 0.05)
    ref = _np(engine.worst_case_sup_batch(dA, dB, 10, 0.03, 0.03, "2"))
    tA, tB = (torch.tensor(a, device=engine.device) for a in (dA, dB))
    G = torch.empty(300, dtype=torch.float64, device=engine.device)
    rc = engine.lib.lqmpc_worst_case_sup_batch(engine._h, 300, _ptr(tA), _ptr(tB), 10, 0.03, 0.03, WORST_NORMS["2"],
                                               200, 1e-8, _ptr(tA), _ptr(tB), _ptr(G), None, None, None, None)
    assert rc == 0
    engine.sync()
    assert np.array_equal(tA.cpu().numpy(), ref["dA"]) and np.array_equal(tB.cpu().numpy(), ref["dB"])
    assert np.array_equal(G.cpu().numpy(), ref["gamma"])
    # every output NULL but one, for each output of the gradient pass
    full = _np(engine.ratio_sup_batch(dA, dB, 10, grad=True))
    tA, tB = (torch.tensor(a, device=engine.device) for a in (dA, dB))
    names = ("gamma", "x_worst", "gap", "rho", "gA", "gB", "flags")
    for i, k in enumerate(names):
        out = torch.zeros_like(torch.as_tensor(full[k], device=engine.device))
        args = [None] * 7
        args[i] = _ptr(out)
        assert engine.lib.lqmpc_ratio_sup_batch(engine._h, 300, _ptr(tA), _ptr(tB), 10, *args) == 0
        engine.sync()
        assert np.array_equal(out.cpu().numpy(), full[k], equal_nan=True), k
    n0 = engine.launch_count
    assert engine.lib.lqmpc_ratio_sup_batch(engine._h, 0, None, None, 10, *[None] * 7) == 0
    assert engine.lib.lqmpc_worst_case_sup_batch(engine._h, 0, None, None, 10, 0.1, 0.1, 0, 200, 1e-8,
                                                 *[None] * 7) == 0
    assert engine.launch_count == n0


def test_error_paths(engine, monkeypatch):
    EINVAL, ESTATE = -1, -4
    pb = synth()
    _set(engine, pb)
    dA, dB = (torch.zeros(k, 4, dtype=torch.float64, device=engine.device) for k in (16, 8))
    p = [_ptr(dA), _ptr(dB)]

    def ratio(N=10, ctx=engine, ops=p):
        return ctx.lib.lqmpc_ratio_sup_batch(ctx._h, 4, *ops, N, *[None] * 7)

    def worst(N=10, eA=0.1, eB=0.1, norm=0, it=200, tol=1e-8, ctx=engine, ops=p):
        return ctx.lib.lqmpc_worst_case_sup_batch(ctx._h, 4, *ops, N, eA, eB, norm, it, tol, *[None] * 7)

    assert ratio(N=0) == EINVAL and ratio(N=-3) == EINVAL
    assert engine.lib.lqmpc_ratio_sup_batch(engine._h, -1, *p, 10, *[None] * 7) == EINVAL
    for ops in ([None, p[1]], [p[0], None]):
        assert ratio(ops=ops) == EINVAL and worst(ops=ops) == EINVAL
    for kw in (dict(N=0), dict(eA=-1e-3), dict(eB=float("inf")), dict(eA=float("nan")), dict(norm=3), dict(norm=-1),
               dict(it=-1), dict(tol=0.0), dict(tol=-1.0), dict(tol=float("nan"))):
        assert worst(**kw) == EINVAL, kw
    assert ratio() == 0 and worst() == 0
    with pytest.raises(ValueError):
        engine.worst_case_sup_batch(dA, dB, 10, 0.1, 0.1, "fro")
    monkeypatch.setenv("LQMPC_FORCE_DYN", "1")
    _set(engine, pb)
    monkeypatch.delenv("LQMPC_FORCE_DYN")
    try:
        assert ratio() == EINVAL
        assert "run-time-dimension" in engine.lib.lqmpc_last_error(engine._h).decode()
        assert worst() == EINVAL
    finally:
        _set(engine, pb)
    assert ratio() == 0
    fresh = Engine(0)
    try:
        assert ratio(ctx=fresh) == ESTATE and worst(ctx=fresh) == ESTATE
        from lq_mpc_b200.sampling import synth_problem
        A4, B4, Q4, R4 = synth_problem(16, 4, seed=0)
        fresh.set_problem_tiled(A4, B4, Q4, R4, Q4, 12)
        assert ratio(ctx=fresh) == EINVAL
        assert "tiled" in fresh.lib.lqmpc_last_error(fresh._h).decode()
        assert worst(ctx=fresh) == EINVAL
        A5, B5, Q5, R5 = synth_problem(5, 2, seed=0)
        fresh.set_problem(A5, B5, Q5, R5)
        assert ratio(ctx=fresh) == EINVAL and worst(ctx=fresh) == EINVAL
        with pytest.raises(EngineError):
            fresh.ratio_sup_batch(np.zeros((25, 2)), np.zeros((10, 2)), 10)
    finally:
        fresh.close()


def test_worst_case_search_sup(engine):
    from lq_mpc_b200.sampling import device_error_grids, synth_problem, synth_samples_soa
    from lq_mpc_b200.worst_case import worst_case_search, worst_case_search_sup
    A, B, Q, R = synth_problem(4, 2, seed=0)
    engine.set_problem(A, B, Q, R, Q, None, None, 0)
    for norm, e in (("max", 0.05), ("f", 0.05)):
        if norm == "max":
            dA, dB, _ = synth_samples_soa(4, 2, 3000, seed=1, e=e)
        else:
            dA, dB = device_error_grids(engine, 4, 2, [e], 600, "f", allow_projected=True)
        r = worst_case_search_sup(engine, dA, dB, 10, e, e, norm, top_k=16)
        assert r["best_ratio"] >= r["sampled_max_ratio"]
        assert r["ratio_start"][0].item() == r["sampled_max_ratio"]
        gamma = engine.ratio_sup_batch(dA, dB, 10)["gamma"].cpu().numpy()
        assert r["sampled_max_ratio"] == gamma.max() and r["sampled_argmax"] == int(np.argmax(gamma))
        gA, gB, xw = r["dA"].cpu().numpy(), r["dB"].cpu().numpy(), r["x_worst"].cpu().numpy()
        for s in range(gA.shape[1]):
            assert feasible(gA[:, s].reshape(4, 4), e, norm) and feasible(gB[:, s].reshape(4, 2), e, norm)
        assert np.all(r["ratio"].cpu().numpy() >= r["ratio_start"].cpu().numpy() * (1 - 1e-12))
        assert np.all(np.isfinite(xw)) and 0 <= r["best_index"] < dA.shape[-1]
        # gamma bounds the ratio at every state: the per-x0 search's sampled maximum at x_worst lies below it
        per = worst_case_search(engine, dA, dB, xw[:, 0], 10, e, e, norm, top_k=16)
        assert per["sampled_max_ratio"] <= r["sampled_max_ratio"] * (1 + 1e-12)
