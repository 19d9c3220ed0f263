"""GPU tier — lqmpc_simulate_inf_grad_batch / lqmpc_worst_case_inf_batch (worst_inf.cuh on the device, k_worst_inf.cu)
on the B200: the input-constrained closed loop's certified J_inf and its gradient in the model error against the CPU-tier
harness (tests/test_inf_grad_host.py) for every compiled (n, m) pair, J_inf / T_cert / flags against
lqmpc_simulate_inf_batch, the ascent against the harness, grid-stride launches, batch sizes, NULL and in-place outputs,
the error paths and worst_case_search_inf on the shipped sweep's inputs."""
import numpy as np
import pytest
import torch

from lq_mpc_b200.engine import FLAG_QP_ACTIVE, WORST_NORMS, Engine, EngineError, _ptr
from oracle import np_oracle as o
from tests.test_inf_grad_host import (COMPILED_DIMS, host_ascent_inf, host_grad_inf, saturating_case)
from tests.test_worst_case_host import feasible

pytestmark = pytest.mark.gpu


def _np(d):
    return {k: (v.cpu().numpy() if isinstance(v, torch.Tensor) else v) for k, v in d.items()}


def _set(engine, pb):
    A, B, Q, R, Pt, lo, hi = pb
    engine.set_problem(A, B, Q, R, Pt, lo, hi, 30)


def _grad_close(d, h, ok, rtol=1e-9):
    """device and harness gradients on the samples `ok`: the device build contracts into FMAs, the harness does not"""
    for s in np.flatnonzero(ok):
        g = np.concatenate([d["gA"][:, s], d["gB"][:, s]])
        hg = np.concatenate([h["gA"][:, s], h["gB"][:, s]])
        assert np.max(np.abs(g - hg)) <= rtol * np.max(np.abs(hg)), s


@pytest.mark.parametrize("n,m", COMPILED_DIMS)
def test_device_vs_harness(engine, n, m):
    checked = 0
    for general in (False, True):
        pb, dA, dB, x0, N = saturating_case(n, m, 2000 + 10 * n + m + 100 * general, S=64, general=general)
        _set(engine, pb)
        d = _np(engine.simulate_inf_grad_batch(dA, dB, N, x0=x0))
        v = _np(engine.simulate_inf_grad_batch(dA, dB, N, x0=x0, grad=False))
        h = host_grad_inf(pb, dA, dB, x0, N)
        for k in ("J_inf", "T_cert", "rho", "flags"):
            assert np.array_equal(v[k], d[k], equal_nan=True), k       # the value-only call: the same value
        assert np.array_equal(d["flags"], h["flags"]) and np.array_equal(d["T_cert"], h["T_cert"])
        ok = (d["flags"] & ~FLAG_QP_ACTIVE) == 0
        assert ok.sum() >= 48 and np.any(d["flags"] & FLAG_QP_ACTIVE)
        assert np.all(np.abs(d["J_inf"][ok] - h["J"][ok]) <= 1e-12 * h["J"][ok])
        assert np.all(np.abs(d["rho"] - h["rho"]) <= 1e-13)
        assert np.all(np.isnan(d["gA"][:, ~ok])) and np.all(np.isnan(d["gB"][:, ~ok]))
        _grad_close(d, h, ok)
        checked += ok.sum()
    assert checked >= 96


@pytest.mark.parametrize("n,m", [(2, 1), (4, 2), (3, 3), (8, 2)])
def test_value_equals_simulate_inf(engine, n, m):
    """J_inf, T_cert and flags are those of lqmpc_simulate_inf_batch bit for bit (the same header code computes them),
    per-sample and shared initial states, including unstable and uncertified samples."""
    pb, dA, dB, x0, N = saturating_case(n, m, 2200 + 10 * n + m, S=500, e=0.2)
    _set(engine, pb)
    for T_max in (1000, 2):
        for kw in (dict(x0=x0), dict(x0_shared=x0[:, 0])):
            ref = _np(engine.simulate_inf_batch(dA, dB, N, T_max, **kw))
            for grad in (True, False):
                d = _np(engine.simulate_inf_grad_batch(dA, dB, N, T_max, grad=grad, **kw))
                assert np.array_equal(d["J_inf"], ref["J_inf"], equal_nan=True)
                assert np.array_equal(d["T_cert"], ref["T_cert"]) and np.array_equal(d["flags"], ref["flags"])


@pytest.mark.parametrize("norm", ["max", "f", "2"])
def test_ascent_on_the_device(engine, norm):
    total = agree = 0
    for (n, m, seed, e) in ((2, 1, 2300, 0.05), (4, 2, 2301, 0.02)):
        pb, dA, dB, x0, N = saturating_case(n, m, seed, S=16, e=e)
        _set(engine, pb)
        got = _np(engine.worst_case_inf_batch(dA, dB, N, e, e, norm, x0=x0))
        start = _np(engine.worst_case_inf_batch(dA, dB, N, e, e, norm, max_iter=0, x0=x0))
        h = host_ascent_inf(pb, dA, dB, x0, N, e, e, norm)
        for s in range(16):
            assert feasible(got["dA"][:, s].reshape(n, n), e, norm) and feasible(got["dB"][:, s].reshape(n, m), e, norm)
        assert np.all(got["J_inf"] >= start["J_inf"])
        fin = np.isfinite(got["J_inf"])
        v = _np(engine.simulate_inf_batch(got["dA"][:, fin], got["dB"][:, fin], N, 1000, x0=x0[:, fin]))
        assert np.array_equal(v["J_inf"], got["J_inf"][fin]) and np.array_equal(v["T_cert"], got["T_cert"][fin])
        both = ((got["flags"] & ~FLAG_QP_ACTIVE) == 0) & ((h["flags"] & ~FLAG_QP_ACTIVE) == 0)
        total += both.sum()
        agree += np.sum(np.abs(got["J_inf"][both] - h["J"][both]) <= 1e-9 * h["J"][both])
    assert total >= 16 and agree >= 0.95 * total


def test_grid_stride_and_permutation(engine, monkeypatch):
    """Two CTAs of 128 threads for 1 500 samples (about 6 per thread): a permuted batch gives permuted results, and
    the same bits as one sample per thread."""
    pb, dA, dB, x0, N = saturating_case(4, 2, 2400, S=1500, e=0.05)
    _set(engine, pb)
    perm = np.random.default_rng(9).permutation(1500)
    calls = (lambda a, b, x: engine.simulate_inf_grad_batch(a, b, N, x0=x),
             lambda a, b, x: engine.simulate_inf_grad_batch(a, b, N, x0=x, grad=False),
             lambda a, b, x: engine.worst_case_inf_batch(a, b, N, 0.05, 0.05, "f", max_iter=10, x0=x))
    monkeypatch.setenv("LQMPC_WORST_CTAS", "2")
    strided = []
    for call in calls:
        r0 = _np(call(dA, dB, x0))
        r1 = _np(call(dA[:, perm], dB[:, perm], x0[:, perm]))
        for k, v in r0.items():
            assert np.array_equal(v[..., perm], r1[k], equal_nan=v.dtype.kind == "f"), k
        strided.append(r0)
    monkeypatch.delenv("LQMPC_WORST_CTAS")
    for call, r0 in zip(calls, strided):
        full = _np(call(dA, dB, x0))
        assert all(np.array_equal(full[k], r0[k], equal_nan=True) for k in r0)


@pytest.mark.parametrize("S", [1, 127, 129])
def test_batch_sizes(engine, S):
    pb, dA, dB, x0, N = saturating_case(3, 2, 2500 + S, S=S)
    _set(engine, pb)
    d = _np(engine.simulate_inf_grad_batch(dA, dB, N, x0=x0))
    h = host_grad_inf(pb, dA, dB, x0, N)
    ok = (h["flags"] & ~FLAG_QP_ACTIVE) == 0
    assert np.array_equal(d["flags"], h["flags"]) and ok.sum() >= 0.9 * S
    assert np.all(np.abs(d["J_inf"][ok] - h["J"][ok]) <= 1e-12 * h["J"][ok])
    _grad_close(d, h, ok)
    w = _np(engine.worst_case_inf_batch(dA, dB, N, 0.01, 0.01, "max", x0=x0))
    assert np.all(np.abs(w["dA"]) <= 0.01) and np.all(w["J_inf"][ok] >= d["J_inf"][ok])


def test_null_and_in_place_outputs_and_empty_batch(engine):
    pb, dA, dB, x0, N = saturating_case(4, 2, 2600, S=300, e=0.03)
    _set(engine, pb)
    ref = _np(engine.worst_case_inf_batch(dA, dB, N, 0.03, 0.03, "2", x0=x0))
    tA, tB, tx = (torch.tensor(a, device=engine.device) for a in (dA, dB, x0))
    J = torch.empty(300, dtype=torch.float64, device=engine.device)
    rc = engine.lib.lqmpc_worst_case_inf_batch(engine._h, 300, _ptr(tA), _ptr(tB), N, 1000, None, _ptr(tx), 0.03, 0.03,
                                               WORST_NORMS["2"], 200, 1e-8, _ptr(tA), _ptr(tB), _ptr(J), None, None,
                                               None, None)
    assert rc == 0
    engine.sync()
    assert np.array_equal(tA.cpu().numpy(), ref["dA"]) and np.array_equal(tB.cpu().numpy(), ref["dB"])
    assert np.array_equal(J.cpu().numpy(), ref["J_inf"], equal_nan=True)
    # every output NULL but one, for each output of the gradient pass
    full = _np(engine.simulate_inf_grad_batch(dA, dB, N, x0=x0))
    tA, tB = (torch.tensor(a, device=engine.device) for a in (dA, dB))
    names = ("J_inf", "T_cert", "rho", "gA", "gB", "flags")
    for i, k in enumerate(names):
        out = torch.zeros_like(torch.as_tensor(full[k], device=engine.device))
        args = [None] * 6
        args[i] = _ptr(out)
        assert engine.lib.lqmpc_simulate_inf_grad_batch(engine._h, 300, _ptr(tA), _ptr(tB), N, 1000, None, _ptr(tx),
                                                        *args) == 0
        engine.sync()
        assert np.array_equal(out.cpu().numpy(), full[k], equal_nan=True), k
    n0 = engine.launch_count
    assert engine.lib.lqmpc_simulate_inf_grad_batch(engine._h, 0, None, None, N, 1000, None, _ptr(tx),
                                                    *[None] * 6) == 0
    assert engine.lib.lqmpc_worst_case_inf_batch(engine._h, 0, None, None, N, 1000, None, _ptr(tx), 0.1, 0.1, 0, 200,
                                                 1e-8, *[None] * 7) == 0
    assert engine.launch_count == n0


def test_error_paths(engine, monkeypatch):
    EINVAL, ESTATE = -1, -4
    pb, _, _, _, _ = saturating_case(4, 2, 2700)
    _set(engine, pb)
    dA, dB, x0 = (torch.zeros(k, 4, dtype=torch.float64, device=engine.device) for k in (16, 8, 4))
    xs = torch.zeros(4, dtype=torch.float64, device=engine.device)
    p = [_ptr(dA), _ptr(dB)]

    def grad(N=10, T_max=100, x=(None, _ptr(x0)), ctx=engine, ops=p):
        return ctx.lib.lqmpc_simulate_inf_grad_batch(ctx._h, 4, *ops, N, T_max, *x, *[None] * 6)

    def worst(N=10, T_max=100, x=(None, _ptr(x0)), eA=0.1, eB=0.1, norm=0, it=200, tol=1e-8, ctx=engine, ops=p):
        return ctx.lib.lqmpc_worst_case_inf_batch(ctx._h, 4, *ops, N, T_max, *x, eA, eB, norm, it, tol, *[None] * 7)

    for kw in (dict(N=0), dict(N=-3), dict(T_max=-1), dict(x=(None, None)), dict(x=(_ptr(xs), _ptr(x0))),
               dict(ops=[None, p[1]]), dict(ops=[p[0], None])):
        assert grad(**kw) == EINVAL and worst(**kw) == EINVAL, kw
    assert engine.lib.lqmpc_simulate_inf_grad_batch(engine._h, -1, *p, 10, 100, None, _ptr(x0), *[None] * 6) == EINVAL
    for kw in (dict(eA=-1e-3), dict(eB=float("inf")), dict(eA=float("nan")), dict(norm=3), dict(norm=-1),
               dict(it=-1), dict(tol=0.0), dict(tol=-1.0), dict(tol=float("nan"))):
        assert worst(**kw) == EINVAL, kw
    assert grad() == 0 and worst() == 0 and grad(x=(_ptr(xs), None)) == 0
    with pytest.raises(ValueError):
        engine.worst_case_inf_batch(dA, dB, 10, 0.1, 0.1, "fro", x0=x0)
    # references and an input polytope are refused
    engine.set_references(np.full((4, 10), 0.1), np.full((2, 10), 0.1))
    try:
        assert grad() == EINVAL and "references" in engine.lib.lqmpc_last_error(engine._h).decode()
        assert worst() == EINVAL
    finally:
        _set(engine, pb)
    engine.set_input_polytope(np.array([[1.0, 0.0], [-1.0, 0.0], [0.0, 1.0], [0.0, -1.0]]) * 4)
    try:
        assert grad() == EINVAL and "polytope" in engine.lib.lqmpc_last_error(engine._h).decode()
        assert worst() == EINVAL
    finally:
        _set(engine, pb)
    assert grad() == 0
    monkeypatch.setenv("LQMPC_FORCE_DYN", "1")
    _set(engine, pb)
    monkeypatch.delenv("LQMPC_FORCE_DYN")
    try:
        assert grad() == EINVAL and "run-time-dimension" in engine.lib.lqmpc_last_error(engine._h).decode()
        assert worst() == EINVAL
    finally:
        _set(engine, pb)
    fresh = Engine(0)
    try:
        assert grad(ctx=fresh) == ESTATE and worst(ctx=fresh) == ESTATE
        from lq_mpc_b200.sampling import synth_problem
        A4, B4, Q4, R4 = synth_problem(16, 4, seed=0)
        fresh.set_problem_tiled(A4, B4, Q4, R4, Q4, 12)
        assert grad(ctx=fresh) == EINVAL and "tiled" in fresh.lib.lqmpc_last_error(fresh._h).decode()
        assert worst(ctx=fresh) == EINVAL
        A5, B5, Q5, R5 = synth_problem(5, 2, seed=0)
        fresh.set_problem(A5, B5, Q5, R5)
        assert grad(ctx=fresh) == EINVAL and worst(ctx=fresh) == EINVAL
        with pytest.raises(EngineError):
            fresh.simulate_inf_grad_batch(np.zeros((25, 2)), np.zeros((10, 2)), 10, x0_shared=np.ones(5))
    finally:
        fresh.close()


def test_worst_case_search_inf_on_the_shipped_sweep(engine, golden, example):
    """The 2-state sweep's inputs (error level 4 of the Frobenius grids, N = 7) with the shipped box and x_start."""
    from lq_mpc_b200.worst_case import worst_case_search_inf
    ex, z = example, golden
    A, B, Q, R, lo, hi = ex["A"], ex["B"], ex["Q"], ex["R"], ex["lo"], ex["hi"]
    engine.set_problem(A, B, Q, R, Q, lo, hi, 30)
    xs = o.circle_generator(8, 1.5, o.local_radius(lo, hi, -o.dlqr(A, B, Q, R)[0], Q), Q)[:, 1]
    eA, eB = z["error_A_f"], z["error_B_f"]
    S = eA.shape[2]
    dA, dB = eA[:, :, :, 4].reshape(4, S), eB[:, :, :, 4].reshape(2, S)
    e_A = float(np.max(np.linalg.norm(eA[:, :, :, 4], axis=(0, 1))))
    e_B = float(np.max(np.linalg.norm(eB[:, :, :, 4], axis=(0, 1))))
    r = worst_case_search_inf(engine, dA, dB, 7, e_A, e_B, "f", x0_shared=xs, top_k=16)
    J = engine.simulate_inf_batch(dA, dB, 7, 1000, x0_shared=xs)["J_inf"].cpu().numpy()
    assert r["n_uncertified"] == 0 and r["sampled_max_J"] == J.max() and r["sampled_argmax"] == int(np.argmax(J))
    assert r["J_start"][0].item() == r["sampled_max_J"] and r["best_J"] >= r["sampled_max_J"]
    Jr, Js = r["J"].cpu().numpy(), r["J_start"].cpu().numpy()
    assert np.all(Jr >= Js) and np.all(np.isfinite(Jr)) and r["n_unstable"] == 0
    gA, gB = r["dA"].cpu().numpy(), r["dB"].cpu().numpy()
    for s in range(16):
        assert feasible(gA[:, s].reshape(2, 2), e_A, "f") and feasible(gB[:, s].reshape(2, 1), e_B, "f")
    assert 0 <= r["best_index"] < S and np.all(r["T_cert"].cpu().numpy() >= 0)
