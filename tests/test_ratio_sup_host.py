"""CPU tier — the worst performance ratio over every initial state, gamma(dA, dB) = sup_x x'S x / x'P_exp x =
lambda_max(L^-1 S L^-T), its worst state, eigengap and gradient, and the projected ascent of gamma (worst.cuh's SUP
mode of worst_eval / worst_ascent) compiled with g++ from the engine headers (tests/hostmath/sup.cpp, built like
tests/hostmath/worst.cpp), against scipy's generalized symmetric eigensolver, a torch float64 autograd oracle through
torch.linalg.eigvalsh, 50-digit central differences, and the per-x0 harness of tests/test_worst_case_host.py. The GPU
tier (tests/test_ratio_sup.py) runs the device kernels against this harness."""
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import pytest
import scipy.linalg as sla
import torch

from tests.test_worst_case_host import (COMPILED_DIMS, FLAG_ASCENT_MAXITER, FLAG_UNSTABLE, N_OPC, NORMS, ascent_cases,
                                        closed_loop_rho, feasible, host_ascent, host_grad, plant, project,
                                        samples)

HERE = os.path.dirname(os.path.abspath(__file__))
HM = os.path.join(HERE, "hostmath")
CSRC = os.path.join(os.path.dirname(HERE), "lq_mpc_b200", "csrc")

_P = ctypes.POINTER(ctypes.c_double)
_I = ctypes.POINTER(ctypes.c_int32)
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(HM, "_build")
        os.makedirs(out, exist_ok=True)
        so = os.path.join(out, "libsup.so")
        src = os.path.join(HM, "sup.cpp")
        h = hashlib.sha256()
        for d in [src] + [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith(".cuh")]:
            h.update(open(d, "rb").read())
        stamp = so + ".stamp"
        if not (os.path.exists(so) and os.path.exists(stamp) and open(stamp).read() == h.hexdigest()):
            cmd = ["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-x", "c++", src, "-o", so,
                   "-lm"]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError("g++ failed:\n" + r.stderr)
            open(stamp, "w").write(h.hexdigest())
        _lib = ctypes.CDLL(so)
    return _lib


def _c(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _p(a):
    return a.ctypes.data_as(_P)


def host_sup(pb, dA, dB, N, grad=True):
    """Harness gamma pass: dict gamma, gap, rho [S], x_worst [n][S], flags [S], and gA [n*n][S], gB [n*m][S] with
    grad (grad=False: the value-only call)."""
    A, B, Q, R, Pt = pb
    n, m = B.shape
    S = dA.shape[1]
    keep = [_c(a) for a in (A, B, Q, R, Pt, dA, dB)]
    o = {k: np.zeros(S) for k in ("gamma", "gap", "rho")}
    o["x_worst"], o["flags"] = np.zeros((n, S)), np.zeros(S, dtype=np.int32)
    o["gA"], o["gB"] = (np.zeros((n * n, S)), np.zeros((n * m, S))) if grad else (None, None)
    gp = [_p(o["gA"]), _p(o["gB"])] if grad else [None, None]
    rc = lib().sup_ratio(n, m, *[_p(a) for a in keep[:5]], N_OPC, ctypes.c_int64(S), _p(keep[5]), _p(keep[6]), N,
                         _p(o["gamma"]), _p(o["x_worst"]), _p(o["gap"]), _p(o["rho"]), *gp,
                         o["flags"].ctypes.data_as(_I))
    assert rc == 0
    return o


def host_sup_ascent(pb, dA, dB, N, eA, eB, norm, max_iter=200, tol=1e-8):
    """Harness ascent of gamma: dict dA, dB, gamma, x_worst, rho, iters, flags."""
    A, B, Q, R, Pt = pb
    n, m = B.shape
    S = dA.shape[1]
    keep = [_c(a) for a in (A, B, Q, R, Pt, dA, dB)]
    o = {"dA": np.zeros((n * n, S)), "dB": np.zeros((n * m, S)), "gamma": np.zeros(S), "x_worst": np.zeros((n, S)),
         "rho": np.zeros(S), "iters": np.zeros(S, dtype=np.int32), "flags": np.zeros(S, dtype=np.int32)}
    rc = lib().sup_ascent(n, m, *[_p(a) for a in keep[:5]], N_OPC, ctypes.c_int64(S), _p(keep[5]), _p(keep[6]), N,
                          ctypes.c_double(eA), ctypes.c_double(eB), NORMS[norm], max_iter, ctypes.c_double(tol),
                          _p(o["dA"]), _p(o["dB"]), _p(o["gamma"]), _p(o["x_worst"]), _p(o["rho"]),
                          o["iters"].ctypes.data_as(_I), o["flags"].ctypes.data_as(_I))
    assert rc == 0
    return o


# ---------------------------------------------------------------------------------------------------- the oracle
def pexp(pb):
    """The expert matrix as the engine prepares it: N_OPC Riccati steps from P_t on the true model."""
    A, B, Q, R, Pt = pb
    P = Pt
    for _ in range(N_OPC):
        P = Q + A.T @ (P - P @ B @ np.linalg.solve(R + B.T @ P @ B, B.T @ P)) @ A
    return (P + P.T) / 2


def oracle_S(pb, dA, dB, N):
    """The closed-loop cost matrix S in torch float64 (S = W + A_cl'S A_cl by the Kronecker system); dA (n, n),
    dB (n, m) may require grad."""
    A, B, Q, R, Pt = (torch.as_tensor(a, dtype=torch.float64) for a in pb)
    n = A.shape[0]
    Ah, Bh, P = A + dA, B + dB, Pt
    for k in range(N):
        G = R + Bh.T @ P @ Bh
        K = -torch.linalg.solve(G, Bh.T @ P @ Ah)
        if k < N - 1:
            P = Q + Ah.T @ (P - P @ Bh @ torch.linalg.solve(G, Bh.T @ P)) @ Ah
    Acl, W = A + B @ K, Q + K.T @ R @ K
    S = torch.linalg.solve(torch.eye(n * n, dtype=torch.float64) - torch.kron(Acl.T, Acl.T), W.reshape(-1))
    S = S.reshape(n, n)
    return (S + S.T) / 2


def oracle_gamma(pb, dA, dB, N):
    Li = torch.linalg.inv(torch.linalg.cholesky(torch.as_tensor(pexp(pb))))
    return torch.linalg.eigvalsh(Li @ oracle_S(pb, dA, dB, N) @ Li.T)[-1]


def oracle_gamma_grad(pb, dA, dB, N):
    tA = torch.tensor(dA, dtype=torch.float64, requires_grad=True)
    tB = torch.tensor(dB, dtype=torch.float64, requires_grad=True)
    g = oracle_gamma(pb, tA, tB, N)
    g.backward()
    return g.item(), tA.grad.numpy(), tB.grad.numpy()


def sup_residual(pb, dA, dB, N, eA, eB, norm):
    """r = ||Proj(u + g^/||g^||) - u||_2 in u = (dA/eA, dB/eB), with the autograd gradient of gamma."""
    _, gA, gB = oracle_gamma_grad(pb, dA, dB, N)
    gn = np.sqrt(eA ** 2 * np.sum(gA ** 2) + eB ** 2 * np.sum(gB ** 2))
    if gn == 0:
        return 0.0
    r2 = 0.0
    for M, g, e in ((dA, gA, eA), (dB, gB, eB)):
        if e > 0:
            r2 += np.sum((project(M + e * e * g / gn, e, norm) - M) ** 2) / e ** 2
    return float(np.sqrt(r2))


# ---------------------------------------------------------------------------------------------------- 1. value
@pytest.mark.parametrize("n,m", COMPILED_DIMS)
def test_value_worst_state_and_gradient(n, m):
    rng = np.random.default_rng(700 + 10 * n + m)
    checked = grads = 0
    for N, general in ((1, False), (5, True), (10, True), (30, False)):
        pb = plant(rng, n, m, rho=rng.uniform(0.8, 1.05), scalar=not general, general_P=general)
        P = pexp(pb)
        dA, dB, _ = samples(rng, n, m, 4, 0.02)
        h = host_sup(pb, dA, dB, N)
        v = host_sup(pb, dA, dB, N, grad=False)
        for k in ("gamma", "gap", "rho", "x_worst", "flags"):
            assert np.array_equal(v[k], h[k], equal_nan=True), k     # the value-only call computes the same value
        for s in range(4):
            a, b = dA[:, s].reshape(n, n), dB[:, s].reshape(n, m)
            if h["flags"][s] & FLAG_UNSTABLE:
                assert np.isinf(h["gamma"][s]) and np.all(np.isnan(h["x_worst"][:, s])) and np.isnan(h["gap"][s])
                assert np.all(np.isnan(h["gA"][:, s])) and closed_loop_rho(pb, a, b, N) >= 1 - 1e-12
                continue
            assert h["flags"][s] == 0
            S = oracle_S(pb, torch.tensor(a), torch.tensor(b), N).numpy()
            lam = sla.eigh(S, P, eigvals_only=True)
            g = h["gamma"][s]
            assert abs(g - lam[-1]) <= 1e-11 * abs(lam[-1]), (N, s)
            gap = 1.0 if n == 1 else (lam[-1] - lam[-2]) / lam[-1]
            assert abs(h["gap"][s] - gap) <= 1e-9
            x = h["x_worst"][:, s]
            assert abs(x @ P @ x - 1) <= 1e-13
            big = np.argmax(np.abs(x))
            assert x[big] > 0
            assert abs((x @ S @ x) / (x @ P @ x) - g) <= 1e-12 * g
            X = rng.normal(size=(n, 1000))
            ratios = np.einsum("is,ij,js->s", X, S, X) / np.einsum("is,ij,js->s", X, P, X)
            assert np.all(ratios <= g * (1 + 1e-12))
            checked += 1
            if h["gap"][s] >= 1e-3:
                _, gA, gB = oracle_gamma_grad(pb, a, b, N)
                ref = np.concatenate([gA.ravel(), gB.ravel()])
                got = np.concatenate([h["gA"][:, s], h["gB"][:, s]])
                assert np.max(np.abs(got - ref)) <= 1e-9 * np.max(np.abs(ref)), (N, s)
                grads += 1
    assert checked >= 10 and grads >= (8 if n > 1 else 10)


def test_scalar_gamma_is_the_ratio_at_x0_one():
    rng = np.random.default_rng(4)
    for N in (1, 3, 10):
        pb = plant(rng, 1, 1, rho=0.95, scalar=False, general_P=True)
        dA, dB, _ = samples(rng, 1, 1, 16, 0.05)
        h = host_sup(pb, dA, dB, N)
        r = host_grad(pb, dA, dB, np.ones((1, 16)), N)
        ok = h["flags"] == 0
        assert ok.sum() >= 8 and np.array_equal(h["flags"], r["flags"])
        assert np.all(np.abs(h["gamma"][ok] - r["ratio"][ok]) <= 1e-14 * r["ratio"][ok])
        assert np.all(h["x_worst"][0, ok] > 0) and np.all(h["gap"][ok] == 1.0)


def test_gradient_near_instability_vs_mpmath():
    """rho(A_cl) > 0.99: 50-digit central differences of gamma, tolerance scaled by 1 / (1 - rho)."""
    import mpmath as mp
    mp.mp.dps = 50
    n, m, N = 2, 1, 6
    A = np.array([[1.02, 0.3], [0.0, 0.97]])
    B = np.array([[0.0], [0.05]])
    Q, R = np.eye(2), np.array([[4.0]])
    pb = (A, B, Q, R, Q)
    rng = np.random.default_rng(7)
    dA, dB, _ = samples(rng, n, m, 3, 0.002)
    h = host_sup(pb, dA, dB, N)
    Am, Bm, Qm, Rm = mp.matrix(A.tolist()), mp.matrix(B.tolist()), mp.matrix(Q.tolist()), mp.matrix(R.tolist())
    Pe = Qm
    for _ in range(N_OPC):
        Pe = Qm + Am.T * (Pe - Pe * Bm * mp.inverse(Rm + Bm.T * Pe * Bm) * Bm.T * Pe) * Am
    Li = mp.inverse(mp.cholesky((Pe + Pe.T) / 2))

    def gamma_mp(a, b):
        Ah, Bh, P = Am + a, Bm + b, Qm
        for k in range(N):
            Gi = mp.inverse(Rm + Bh.T * P * Bh)
            K = -(Gi * (Bh.T * P * Ah))
            if k < N - 1:
                P = Qm + Ah.T * (P - P * Bh * Gi * Bh.T * P) * Ah
        Acl, W = Am + Bm * K, Qm + K.T * Rm * K
        M = mp.eye(n * n)
        for i in range(n):
            for j in range(n):
                for k in range(n):
                    for l in range(n):
                        M[i * n + j, k * n + l] -= Acl[k, i] * Acl[l, j]
        Sv = mp.lu_solve(M, mp.matrix([W[i, j] for i in range(n) for j in range(n)]))
        S = mp.matrix(n, n)
        for i in range(n):
            for j in range(n):
                S[i, j] = (Sv[i * n + j] + Sv[j * n + i]) / 2
        C = Li * S * Li.T
        C = (C + C.T) / 2
        return max(mp.eigsy(C, eigvals_only=True))

    done = 0
    for s in range(3):
        rho = closed_loop_rho(pb, dA[:, s].reshape(n, n), dB[:, s].reshape(n, m), N)
        assert 0.99 < rho < 1 and h["flags"][s] == 0 and h["gap"][s] >= 1e-3
        a0, b0 = mp.matrix(dA[:, s].reshape(n, n).tolist()), mp.matrix(dB[:, s].reshape(n, m).tolist())
        assert abs(float(gamma_mp(a0, b0)) - h["gamma"][s]) <= 1e-11 / (1 - rho) * h["gamma"][s]
        hh = mp.mpf("1e-20")
        g = []
        for blk, shape in ((0, (n, n)), (1, (n, m))):
            for i in range(shape[0]):
                for j in range(shape[1]):
                    ap, am_, bp, bm = a0.copy(), a0.copy(), b0.copy(), b0.copy()
                    if blk == 0:
                        ap[i, j] += hh; am_[i, j] -= hh
                    else:
                        bp[i, j] += hh; bm[i, j] -= hh
                    g.append(float((gamma_mp(ap, bp) - gamma_mp(am_, bm)) / (2 * hh)))
        g = np.array(g)
        hg = np.concatenate([h["gA"][:, s], h["gB"][:, s]])
        assert np.max(np.abs(hg - g)) <= 1e-11 / (1 - rho) * np.max(np.abs(g))
        done += 1
    assert done == 3


# ---------------------------------------------------------------------------------------------------- 2. ascent
def check_sup_ascent(pb, dA, dB, N, eA, eB, norm, got, start_gamma, tol=1e-8):
    """Feasibility, gamma >= the projected start's gamma, gamma against the oracle at the returned point, the
    residual with the autograd gradient of gamma (where the top eigenvalue is simple); returns the number of
    converged entries checked."""
    n, m = pb[1].shape
    conv = 0
    for s in range(dA.shape[1]):
        a, b = got["dA"][:, s].reshape(n, n), got["dB"][:, s].reshape(n, m)
        assert feasible(a, eA, norm) and feasible(b, eB, norm), s
        assert got["gamma"][s] >= start_gamma[s], s
        if got["flags"][s] & FLAG_UNSTABLE:
            assert np.isinf(got["gamma"][s]) and closed_loop_rho(pb, a, b, N) >= 1 - 1e-12
            continue
        g = float(oracle_gamma(pb, torch.tensor(a), torch.tensor(b), N))
        assert abs(got["gamma"][s] - g) <= 1e-11 * g, s
        if not got["flags"][s] & FLAG_ASCENT_MAXITER:
            assert got["flags"][s] == 0
            gap = host_sup(pb, got["dA"][:, s:s + 1], got["dB"][:, s:s + 1], N, grad=False)["gap"][0]
            if gap >= 1e-6:
                assert sup_residual(pb, a, b, N, eA, eB, norm) <= tol + 1e-8, s
                conv += 1
    return conv


@pytest.mark.parametrize("norm", ["max", "f", "2"])
def test_ascent(norm):
    conv = 0
    for pb, dA, dB, _, N, eA, eB in ascent_cases():
        got = host_sup_ascent(pb, dA, dB, N, eA, eB, norm)
        start = host_sup_ascent(pb, dA, dB, N, eA, eB, norm, max_iter=0)
        conv += check_sup_ascent(pb, dA, dB, N, eA, eB, norm, got, start["gamma"])
        assert np.all(got["iters"] >= 1)
    assert conv >= 4


@pytest.mark.parametrize("norm", ["max", "f", "2"])
def test_ascent_is_jointly_stationary(norm):
    """At a converged gamma ascent with a simple top eigenvalue, (dA, dB, x_worst) is stationary for J / V_expert over
    (dA, dB, x0): the per-x0 ascent from (dA, dB) at x0 = x_worst raises the ratio by at most 1e-9 relative."""
    done = 0
    for pb, dA, dB, _, N, eA, eB in ascent_cases():
        got = host_sup_ascent(pb, dA, dB, N, eA, eB, norm)
        gap = host_sup(pb, got["dA"], got["dB"], N, grad=False)["gap"]
        sel = np.flatnonzero((got["flags"] == 0) & (gap >= 1e-6))
        if len(sel) == 0:
            continue
        per = host_ascent(pb, got["dA"][:, sel], got["dB"][:, sel], got["x_worst"][:, sel], N, eA, eB, norm)
        ok = per["flags"] == 0
        assert np.all(per["ratio"][ok] <= got["gamma"][sel][ok] * (1 + 1e-9))
        assert np.all(per["ratio"] >= got["gamma"][sel] * (1 - 1e-12))
        done += ok.sum()
    assert done >= 4


def test_scalar_box_matches_the_per_x0_ascent():
    """n = m = 1 (the case of the per-x0 grid search): gamma = J(x0 = 1) / P_exp, so both ascents agree."""
    A, B, Q, R = np.array([[1.1]]), np.array([[0.8]]), np.array([[1.0]]), np.array([[0.5]])
    pb, N, e = (A, B, Q, R, Q), 3, 0.2
    s = np.linspace(-e, e, 5)
    dA, dB = np.repeat(s, 5)[None, :], np.tile(s, 5)[None, :]
    got = host_sup_ascent(pb, dA, dB, N, e, e, "max")
    ref = host_ascent(pb, dA, dB, np.ones((1, 25)), N, e, e, "max")
    assert np.all(got["flags"] == 0) and np.all(ref["flags"] == 0)
    assert np.all(np.abs(got["gamma"] - ref["ratio"]) <= 1e-9 * ref["ratio"])
    assert abs(got["gamma"].max() - ref["ratio"].max()) <= 1e-9 * ref["ratio"].max()


def test_ascent_finds_a_destabilising_error():
    """The case of the per-x0 test, without an x0: every start is stable, the set holds a destabilising error."""
    A, B, Q, R = np.array([[1.3, 0.2], [0.0, 0.9]]), np.array([[1.0], [0.3]]), np.eye(2), np.eye(1)
    pb, N, e = (A, B, Q, R, Q), 8, 0.35
    dA, dB, _ = samples(np.random.default_rng(2), 2, 1, 8, 0.02)
    assert np.all(host_sup(pb, dA, dB, N)["flags"] == 0)
    for norm in ("max", "f"):
        got = host_sup_ascent(pb, dA, dB, N, e, e, norm)
        hit = np.flatnonzero(got["flags"] & FLAG_UNSTABLE)
        assert len(hit) >= 1
        for s in hit:
            assert np.isinf(got["gamma"][s]) and np.all(np.isnan(got["x_worst"][:, s]))
            a, b = got["dA"][:, s].reshape(2, 2), got["dB"][:, s].reshape(2, 1)
            assert feasible(a, e, norm) and feasible(b, e, norm)
            assert closed_loop_rho(pb, a, b, N) >= 1 - 1e-12
