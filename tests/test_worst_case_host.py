"""CPU tier — the gradient of the unconstrained law's J_inf in the model error and the projected ascent over the error
set (worst.cuh: worst_eval / worst_ascent) compiled with g++ from the engine headers (tests/hostmath/worst.cpp, the
flags of tests/hostmath/build.py), against a torch float64 autograd oracle of the same cost: the Riccati recursion
through torch.linalg.solve and S from the Kronecker system. The GPU tier (tests/test_worst_case.py) runs the device
kernels against this harness and the oracle."""
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import pytest
import scipy.linalg as sla
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
HM = os.path.join(HERE, "hostmath")
CSRC = os.path.join(os.path.dirname(HERE), "lq_mpc_b200", "csrc")
COMPILED_DIMS = [(1, 1), (2, 1), (2, 2), (3, 1), (3, 2), (3, 3), (4, 1), (4, 2), (4, 4), (6, 2), (8, 2)]
FLAG_UNSTABLE, FLAG_ASCENT_MAXITER = 1, 2048
NORMS = {"f": 0, "2": 1, "max": 2}
N_OPC = 30

_P = ctypes.POINTER(ctypes.c_double)
_I = ctypes.POINTER(ctypes.c_int32)
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(HM, "_build")
        os.makedirs(out, exist_ok=True)
        so = os.path.join(out, "libworst.so")
        src = os.path.join(HM, "worst.cpp")
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


def host_grad(pb, dA, dB, x0, N):
    """Harness gradient pass: dict J, rho, ratio [S], gA [n*n][S], gB [n*m][S], flags [S] (SoA operands)."""
    A, B, Q, R, Pt = pb
    n, m = B.shape
    S = dA.shape[1]
    keep = [_c(a) for a in (A, B, Q, R, Pt, dA, dB, x0)]
    o = {k: np.zeros(S) for k in ("J", "rho", "ratio")}
    o["gA"], o["gB"], o["flags"] = np.zeros((n * n, S)), np.zeros((n * m, S)), np.zeros(S, dtype=np.int32)
    rc = lib().worst_grad(n, m, *[_p(a) for a in keep[:5]], N_OPC, ctypes.c_int64(S), *[_p(a) for a in keep[5:]], N,
                          _p(o["J"]), _p(o["rho"]), _p(o["ratio"]), _p(o["gA"]), _p(o["gB"]),
                          o["flags"].ctypes.data_as(_I))
    assert rc == 0
    return o


def host_ascent(pb, dA, dB, x0, N, eA, eB, norm, max_iter=200, tol=1e-8):
    """Harness ascent: dict dA, dB, J, rho, ratio, iters, flags."""
    A, B, Q, R, Pt = pb
    n, m = B.shape
    S = dA.shape[1]
    keep = [_c(a) for a in (A, B, Q, R, Pt, dA, dB, x0)]
    o = {"dA": np.zeros((n * n, S)), "dB": np.zeros((n * m, S)), "J": np.zeros(S), "rho": np.zeros(S),
         "ratio": np.zeros(S), "iters": np.zeros(S, dtype=np.int32), "flags": np.zeros(S, dtype=np.int32)}
    rc = lib().worst_ascent(n, m, *[_p(a) for a in keep[:5]], N_OPC, ctypes.c_int64(S), *[_p(a) for a in keep[5:]],
                            N, ctypes.c_double(eA), ctypes.c_double(eB), NORMS[norm], max_iter, ctypes.c_double(tol),
                            _p(o["dA"]), _p(o["dB"]), _p(o["J"]), _p(o["rho"]), _p(o["ratio"]),
                            o["iters"].ctypes.data_as(_I), o["flags"].ctypes.data_as(_I))
    assert rc == 0
    return o


# ---------------------------------------------------------------------------------------------------- the oracle
def oracle_J(pb, dA, dB, x0, N):
    """J_inf in torch float64; dA (n, n), dB (n, m) may require grad."""
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
    x = torch.as_tensor(x0, dtype=torch.float64)
    return x @ S.reshape(n, n) @ x


def oracle_grad(pb, dA, dB, x0, N):
    tA = torch.tensor(dA, dtype=torch.float64, requires_grad=True)
    tB = torch.tensor(dB, dtype=torch.float64, requires_grad=True)
    J = oracle_J(pb, tA, tB, x0, N)
    J.backward()
    return J.item(), tA.grad.numpy(), tB.grad.numpy()


def closed_loop_rho(pb, dA, dB, N):
    A, B, Q, R, Pt = pb
    Ah, Bh, P = A + dA, B + dB, Pt
    for k in range(N):
        G = R + Bh.T @ P @ Bh
        K = -np.linalg.solve(G, Bh.T @ P @ Ah)
        P = Q + Ah.T @ (P - P @ Bh @ np.linalg.solve(G, Bh.T @ P)) @ Ah
    return float(np.max(np.abs(np.linalg.eigvals(A + B @ K))))


def project(M, e, norm):
    """Euclidean projection of one block onto {||M|| <= e} (numpy)."""
    if e == 0:
        return np.zeros_like(M)
    if norm == "max":
        return np.clip(M, -e, e)
    if norm == "f":
        f = np.linalg.norm(M)
        return M if f <= e else M * (e / f)
    U, s, Vt = np.linalg.svd(M, full_matrices=False)
    return M if s[0] <= e else (U * np.minimum(s, e)) @ Vt


def residual(pb, dA, dB, x0, N, eA, eB, norm):
    """r = ||Proj(u + g^/||g^||) - u||_2 in u = (dA/eA, dB/eB), with the autograd gradient."""
    _, gA, gB = oracle_grad(pb, dA, dB, x0, N)
    gn = np.sqrt(eA ** 2 * np.sum(gA ** 2) + eB ** 2 * np.sum(gB ** 2))
    if gn == 0:
        return 0.0
    r2 = 0.0
    for M, g, e in ((dA, gA, eA), (dB, gB, eB)):
        if e > 0:
            r2 += np.sum((project(M + e * e * g / gn, e, norm) - M) ** 2) / e ** 2
    return float(np.sqrt(r2))


def feasible(M, e, norm):
    if norm == "max":
        return np.max(np.abs(M)) <= e
    if norm == "f":
        return np.linalg.norm(M) <= e * (1 + 1e-15)
    return np.linalg.norm(M, ord=2) <= e * (1 + 1e-12)


# ---------------------------------------------------------------------------------------------------- problems
def plant(rng, n, m, rho=0.95, scalar=True, general_P=False):
    A = rng.normal(size=(n, n))
    A *= rho / np.max(np.abs(np.linalg.eigvals(A)))
    B = rng.normal(size=(n, m))
    if scalar:
        Q, R = rng.uniform(0.5, 2) * np.eye(n), rng.uniform(0.2, 2) * np.eye(m)
    else:
        Mq, Mr = rng.normal(size=(n, n)), rng.normal(size=(m, m))
        Q, R = Mq @ Mq.T / n + 0.5 * np.eye(n), Mr @ Mr.T / m + 0.3 * np.eye(m)
    if general_P:
        Mp = rng.normal(size=(n, n))
        Pt = Mp @ Mp.T / n + 0.7 * np.eye(n)
    else:
        Pt = Q
    return A, B, Q, R, Pt


def samples(rng, n, m, S, e):
    return rng.uniform(-e, e, (n * n, S)), rng.uniform(-e, e, (n * m, S)), rng.normal(size=(n, S))


def synth():
    from lq_mpc_b200.sampling import synth_problem
    A, B, Q, R = synth_problem(4, 2, seed=0)
    return A, B, Q, R, Q


# ---------------------------------------------------------------------------------------------------- 1. gradient
@pytest.mark.parametrize("n,m", COMPILED_DIMS)
def test_gradient_vs_autograd(n, m):
    rng = np.random.default_rng(100 + 10 * n + m)
    checked = 0
    for N in (1, 2, 10, 30):
        for scalar, general_P in ((True, False), (False, True)):
            pb = plant(rng, n, m, rho=rng.uniform(0.8, 1.05), scalar=scalar, general_P=general_P)
            dA, dB, x0 = samples(rng, n, m, 3, 0.02)
            h = host_grad(pb, dA, dB, x0, N)
            for s in range(3):
                if h["flags"][s]:
                    continue
                J, gA, gB = oracle_grad(pb, dA[:, s].reshape(n, n), dB[:, s].reshape(n, m), x0[:, s], N)
                assert abs(h["J"][s] - J) <= 1e-12 * abs(J)
                g = np.concatenate([gA.ravel(), gB.ravel()])
                hg = np.concatenate([h["gA"][:, s], h["gB"][:, s]])
                assert np.max(np.abs(hg - g)) <= 1e-9 * np.max(np.abs(g)), (N, scalar, s)
                checked += 1
    assert checked >= 20


def test_gradient_near_instability_vs_mpmath():
    """rho(A_cl) > 0.99: 50-digit central differences, tolerance scaled by 1 / (1 - rho)."""
    import mpmath as mp
    mp.mp.dps = 50
    n, m, N = 2, 1, 6
    A = np.array([[1.02, 0.3], [0.0, 0.97]])
    B = np.array([[0.0], [0.05]])
    Q, R = np.eye(2), np.array([[4.0]])
    pb = (A, B, Q, R, Q)
    rng = np.random.default_rng(7)
    dA, dB, x0 = samples(rng, n, m, 3, 0.002)
    h = host_grad(pb, dA, dB, x0, N)

    def J_mp(a, b, x):
        Am, Bm, Qm, Rm = mp.matrix(A.tolist()), mp.matrix(B.tolist()), mp.matrix(Q.tolist()), mp.matrix(R.tolist())
        Ah, Bh, P = Am + a, Bm + b, Qm
        for k in range(N):
            G = Rm + Bh.T * P * Bh
            Gi = mp.inverse(G)
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
        xv = mp.matrix(list(x))
        return sum(xv[i] * Sv[i * n + j] * xv[j] for i in range(n) for j in range(n))

    done = 0
    for s in range(3):
        rho = closed_loop_rho(pb, dA[:, s].reshape(n, n), dB[:, s].reshape(n, m), N)
        assert 0.99 < rho < 1 and h["flags"][s] == 0
        a0, b0 = mp.matrix(dA[:, s].reshape(n, n).tolist()), mp.matrix(dB[:, s].reshape(n, m).tolist())
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
                    g.append(float((J_mp(ap, bp, x0[:, s]) - J_mp(am_, bm, x0[:, s])) / (2 * hh)))
        g = np.array(g)
        hg = np.concatenate([h["gA"][:, s], h["gB"][:, s]])
        assert np.max(np.abs(hg - g)) <= 1e-11 / (1 - rho) * np.max(np.abs(g))
        done += 1
    assert done == 3


def test_gradient_vanishes_at_the_lqr_gain():
    """P_t = DARE(A, B, Q, R), dA = dB = 0: K0 is the LQR gain, optimal for the true plant."""
    rng = np.random.default_rng(3)
    for n, m in ((2, 1), (3, 2), (4, 2)):
        A, B, Q, R, _ = plant(rng, n, m, rho=1.02)
        pb = (A, B, Q, R, sla.solve_discrete_are(A, B, Q, R))
        x0 = rng.normal(size=(n, 1))
        z = host_grad(pb, np.zeros((n * n, 1)), np.zeros((n * m, 1)), x0, 10)
        dA, dB, _ = samples(rng, n, m, 1, 0.01)
        ref = host_grad(pb, dA, dB, x0, 10)
        gz = np.concatenate([z["gA"][:, 0], z["gB"][:, 0]])
        gr = np.concatenate([ref["gA"][:, 0], ref["gB"][:, 0]])
        assert np.linalg.norm(gz) <= 1e-8 * np.linalg.norm(gr)


# ---------------------------------------------------------------------------------------------------- 3. ascent
def check_ascent(pb, dA, dB, x0, N, eA, eB, norm, got, start_J, tol=1e-8):
    """Feasibility, J >= the projected start's J (start_J [S]), J against the oracle at the returned point, the residual
    with the autograd gradient and e = 0 blocks, on one ascent result (dict of SoA arrays); returns the number of
    converged entries checked."""
    n, m = pb[1].shape
    S = dA.shape[1]
    conv = 0
    for s in range(S):
        a, b = got["dA"][:, s].reshape(n, n), got["dB"][:, s].reshape(n, m)
        assert feasible(a, eA, norm) and feasible(b, eB, norm), s
        if eA == 0:
            assert np.all(a == 0)
        if eB == 0:
            assert np.all(b == 0)
        assert got["J"][s] >= start_J[s], s
        if got["flags"][s] & FLAG_UNSTABLE:
            assert np.isinf(got["J"][s]) and closed_loop_rho(pb, a, b, N) >= 1 - 1e-12
            continue
        J = float(oracle_J(pb, torch.tensor(a), torch.tensor(b), x0[:, s], N))
        assert abs(got["J"][s] - J) <= 1e-12 * abs(J), s
        if not got["flags"][s] & FLAG_ASCENT_MAXITER:
            assert got["flags"][s] == 0
            assert residual(pb, a, b, x0[:, s], N, eA, eB, norm) <= tol + 1e-8, s
            conv += 1
    return conv


@pytest.mark.parametrize("norm", ["max", "f", "2"])
def ascent_cases():
    """(problem, dA, dB, x0, N, e_A, e_B) of the ascent checks: the synthetic 4 x 2 plant at two levels (one with an
    e = 0 block) and an open-loop unstable 2 x 1 plant."""
    rng = np.random.default_rng(11)
    out = []
    for (eA, eB) in ((0.05, 0.05), (0.01, 0.0)):
        out.append((synth(), *samples(rng, 4, 2, 6, 2 * eA), 10, eA, eB))
    out.append((plant(np.random.default_rng(5), 2, 1, rho=1.03), *samples(rng, 2, 1, 6, 0.05), 5, 0.05, 0.05))
    return out


@pytest.mark.parametrize("norm", ["max", "f", "2"])
def test_ascent(norm):
    for pb, dA, dB, x0, N, eA, eB in ascent_cases():
        got = host_ascent(pb, dA, dB, x0, N, eA, eB, norm)
        start = host_ascent(pb, dA, dB, x0, N, eA, eB, norm, max_iter=0)
        assert check_ascent(pb, dA, dB, x0, N, eA, eB, norm, got, start["J"]) >= 4
        assert np.all(got["iters"] >= 1)


def test_scalar_box_matches_grid_search():
    """n = m = 1, box: the best ascent from a 5 x 5 grid of starts against a dense grid refined by scipy."""
    from scipy.optimize import minimize
    A, B, Q, R = np.array([[1.1]]), np.array([[0.8]]), np.array([[1.0]]), np.array([[0.5]])
    pb, N, e, x0 = (A, B, Q, R, Q), 3, 0.2, 1.3

    def J(v):
        a, b = A[0, 0] + v[0], B[0, 0] + v[1]
        P = Q[0, 0]
        for k in range(N):
            G = R[0, 0] + b * P * b
            K = -b * P * a / G
            P = Q[0, 0] + a * (P - P * b * b * P / G) * a
        acl = A[0, 0] + B[0, 0] * K
        return x0 * x0 * (Q[0, 0] + R[0, 0] * K * K) / (1 - acl * acl) if abs(acl) < 1 else np.inf

    g = np.linspace(-e, e, 401)
    vals = np.array([[J((a, b)) for b in g] for a in g])
    i, j = np.unravel_index(np.argmax(vals), vals.shape)
    res = minimize(lambda v: -J(v), [g[i], g[j]], bounds=[(-e, e)] * 2, method="L-BFGS-B",
                   options={"ftol": 1e-15, "gtol": 1e-13})
    best = max(-res.fun, vals[i, j])
    s = np.linspace(-e, e, 5)
    dA = np.repeat(s, 5)[None, :]
    dB = np.tile(s, 5)[None, :]
    got = host_ascent(pb, dA, dB, np.full((1, 25), x0), N, e, e, "max")
    assert np.all(got["flags"] == 0)
    assert abs(got["J"].max() - best) <= 1e-9 * best


def test_ascent_finds_a_destabilising_error():
    """Every start is stable but the set holds an error that destabilises the loop: +inf and UNSTABLE."""
    A, B, Q, R = np.array([[1.3, 0.2], [0.0, 0.9]]), np.array([[1.0], [0.3]]), np.eye(2), np.eye(1)
    pb, N, e = (A, B, Q, R, Q), 8, 0.35
    rng = np.random.default_rng(2)
    dA, dB, x0 = samples(rng, 2, 1, 8, 0.02)
    assert np.all(host_grad(pb, dA, dB, x0, N)["flags"] == 0)
    for norm in ("max", "f"):
        got = host_ascent(pb, dA, dB, x0, N, e, e, norm)
        hit = np.flatnonzero(got["flags"] & FLAG_UNSTABLE)
        assert len(hit) >= 1
        for s in hit:
            assert np.isinf(got["J"][s])
            a, b = got["dA"][:, s].reshape(2, 2), got["dB"][:, s].reshape(2, 1)
            assert feasible(a, e, norm) and feasible(b, e, norm)
            assert closed_loop_rho(pb, a, b, N) >= 1 - 1e-12
