"""CPU tier — the gradient of the input-constrained closed loop's certified J_inf in the model error and its projected
ascent (worst_inf.cuh: inf_grad_eval / inf_ascent) compiled with g++ from the engine headers
(tests/hostmath/infgrad.cpp), against a torch float64 autograd oracle of the same closed loop: every pre-certificate
step solves the equality-constrained condensed QP on the active set box_qp finds by a dense torch solve, and the tail
uses K0 from the torch Riccati recursion and S from the Kronecker system. The GPU tier (tests/test_inf_grad.py) runs
the device kernels against this harness."""
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import np_oracle as o
from tests.test_simulate_inf_host import host_inf, plant, saturating_states
from tests.test_worst_case_host import feasible, host_ascent, host_grad, project

HERE = os.path.dirname(os.path.abspath(__file__))
HM = os.path.join(HERE, "hostmath")
CSRC = os.path.join(os.path.dirname(HERE), "lq_mpc_b200", "csrc")
COMPILED_DIMS = [(1, 1), (2, 1), (2, 2), (3, 1), (3, 2), (3, 3), (4, 1), (4, 2), (4, 4), (6, 2), (8, 2)]
FLAG_UNSTABLE, FLAG_QP_ACTIVE, FLAG_QP_MAXITER = 1, 2, 4
FLAG_TAIL_UNCERTIFIED, FLAG_ASCENT_MAXITER = 1024, 2048
NORMS = {"f": 0, "2": 1, "max": 2}

_P = ctypes.POINTER(ctypes.c_double)
_I = ctypes.POINTER(ctypes.c_int32)
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(HM, "_build")
        os.makedirs(out, exist_ok=True)
        so = os.path.join(out, "libinfgrad.so")
        src = os.path.join(HM, "infgrad.cpp")
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
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


def _p(a):
    return None if a is None else a.ctypes.data_as(_P)


def host_grad_inf(pb, dA, dB, x0, N, T_max=1000, grad=True):
    """Harness gradient pass: dict J, T_cert, rho [S], gA [n*n][S], gB [n*m][S], flags [S]. pb = (A, B, Q, R, P, lo,
    hi) (lo = hi = None: no input bounds); SoA operands."""
    A, B, Q, R, Pt, lo, hi = pb
    n, m = B.shape
    S = dA.shape[1]
    keep = [_c(a) for a in (A, B, Q, R, Pt, lo, hi, dA, dB, x0)]
    o_ = {"J": np.zeros(S), "rho": np.zeros(S), "T_cert": np.zeros(S, dtype=np.int32),
          "flags": np.zeros(S, dtype=np.int32)}
    o_["gA"], o_["gB"] = (np.zeros((n * n, S)), np.zeros((n * m, S))) if grad else (None, None)
    rc = lib().infgrad_grad(n, m, *[_p(a) for a in keep[:7]], ctypes.c_int64(S), *[_p(a) for a in keep[7:]], N, T_max,
                            _p(o_["J"]), o_["T_cert"].ctypes.data_as(_I), _p(o_["rho"]), _p(o_["gA"]), _p(o_["gB"]),
                            o_["flags"].ctypes.data_as(_I))
    assert rc == 0
    return o_


def host_ascent_inf(pb, dA, dB, x0, N, eA, eB, norm, max_iter=200, tol=1e-8, T_max=1000):
    """Harness ascent: dict dA, dB, J, T_cert, rho, iters, flags."""
    A, B, Q, R, Pt, lo, hi = pb
    n, m = B.shape
    S = dA.shape[1]
    keep = [_c(a) for a in (A, B, Q, R, Pt, lo, hi, dA, dB, x0)]
    o_ = {"dA": np.zeros((n * n, S)), "dB": np.zeros((n * m, S)), "J": np.zeros(S), "rho": np.zeros(S),
          "T_cert": np.zeros(S, dtype=np.int32), "iters": np.zeros(S, dtype=np.int32),
          "flags": np.zeros(S, dtype=np.int32)}
    rc = lib().infgrad_ascent(n, m, *[_p(a) for a in keep[:7]], ctypes.c_int64(S), *[_p(a) for a in keep[7:]], N,
                              T_max, ctypes.c_double(eA), ctypes.c_double(eB), NORMS[norm], max_iter,
                              ctypes.c_double(tol), _p(o_["dA"]), _p(o_["dB"]), _p(o_["J"]),
                              o_["T_cert"].ctypes.data_as(_I), _p(o_["rho"]), o_["iters"].ctypes.data_as(_I),
                              o_["flags"].ctypes.data_as(_I))
    assert rc == 0
    return o_


# ---------------------------------------------------------------------------------------------------- the oracle
def _condensed_u0(Ah, Bh, Q, R, Pt, x, N, lo, hi):
    """u_0 of the box QP from x, differentiable in (Ah, Bh, x): the active set from box_qp (numpy, detached), then the
    equality-constrained condensed QP by a dense torch solve."""
    n, m = Bh.shape
    H, g, _ = o.condensed_qp(N, Ah.detach().numpy(), Bh.detach().numpy(), Q.numpy(), R.numpy(), Pt.numpy(),
                             x.detach().numpy())
    lo_t, hi_t = np.tile(lo, N), np.tile(hi, N)
    z = o.box_qp(H, g, lo_t, hi_t)
    at_lo = np.abs(z - lo_t) <= 1e-9 * (1 + np.abs(lo_t))
    at_hi = np.abs(z - hi_t) <= 1e-9 * (1 + np.abs(hi_t))
    # the same condensed QP in torch: z'Hz + 2 g'z
    Gam = torch.zeros((N * n, N * m), dtype=torch.float64)
    Phi, M = [], torch.eye(n, dtype=torch.float64)
    for k in range(N):
        M = Ah @ M
        Phi.append(M)
        for j in range(k + 1):
            Gam[k * n:(k + 1) * n, j * m:(j + 1) * m] = torch.linalg.matrix_power(Ah, k - j) @ Bh
    W = torch.block_diag(*([Q] * (N - 1) + [Pt]))
    Ht = torch.block_diag(*([R] * N)) + Gam.T @ W @ Gam
    gt = Gam.T @ W @ torch.cat([P_ @ x for P_ in Phi])
    fx = np.flatnonzero(at_lo | at_hi)
    fr = np.flatnonzero(~(at_lo | at_hi))
    zc = torch.tensor(np.where(at_hi, hi_t, lo_t)[fx], dtype=torch.float64)
    zf = -torch.linalg.solve(Ht[np.ix_(fr, fr)], gt[fr] + Ht[np.ix_(fr, fx)] @ zc)
    z_full = torch.zeros(N * m, dtype=torch.float64)
    z_full = z_full.index_put((torch.as_tensor(fr),), zf).index_put((torch.as_tensor(fx),), zc)
    return z_full[:m], len(fx) > 0


def oracle_J_inf(pb, dA, dB, x0, N, tau):
    """K2c's J_inf in torch float64 with the certified step tau given (the harness's); dA, dB may require grad.
    Returns (J, number of steps with an active bound)."""
    A, B, Q, R, Pt = (torch.as_tensor(a, dtype=torch.float64) for a in pb[:5])
    lo, hi = pb[5], pb[6]
    n = A.shape[0]
    Ah, Bh, P = A + dA, B + dB, Pt
    for k in range(N):
        G = R + Bh.T @ P @ Bh
        K = -torch.linalg.solve(G, Bh.T @ P @ Ah)
        if k < N - 1:
            P = Q + Ah.T @ (P - P @ Bh @ torch.linalg.solve(G, Bh.T @ P)) @ Ah
    Acl, W = A + B @ K, Q + K.T @ R @ K
    S = torch.linalg.solve(torch.eye(n * n, dtype=torch.float64) - torch.kron(Acl.T, Acl.T), W.reshape(-1)).reshape(n, n)
    x = torch.as_tensor(x0, dtype=torch.float64)
    J = torch.zeros((), dtype=torch.float64)
    active = 0
    for _ in range(tau):
        u, act = _condensed_u0(Ah, Bh, Q, R, Pt, x, N, lo, hi)
        active += int(act)
        J = J + x @ Q @ x + u @ R @ u
        x = A @ x + B @ u
    return J + x @ S @ x, active


def oracle_grad_inf(pb, dA, dB, x0, N, tau):
    tA = torch.tensor(dA, dtype=torch.float64, requires_grad=True)
    tB = torch.tensor(dB, dtype=torch.float64, requires_grad=True)
    J, active = oracle_J_inf(pb, tA, tB, x0, N, tau)
    J.backward()
    return J.item(), tA.grad.numpy(), tB.grad.numpy(), active


# ---------------------------------------------------------------------------------------------------- problems
def general_plant(rng, n, m):
    """plant() with general Q, R and a terminal weight P != Q."""
    A, B, _, _, lo, hi = plant(rng, n, m)
    Mq, Mr, Mp = rng.normal(size=(n, n)), rng.normal(size=(m, m)), rng.normal(size=(n, n))
    Q, R, Pt = Mq @ Mq.T / n + 0.5 * np.eye(n), Mr @ Mr.T / m + 0.3 * np.eye(m), Mp @ Mp.T / n + 0.7 * np.eye(n)
    return A, B, Q, R, Pt, lo, hi


def saturating_case(n, m, seed, S=4, general=False, e=0.01, t=(1.5, 3.0)):
    rng = np.random.default_rng(seed)
    if general:
        pb = general_plant(rng, n, m)
    else:
        A, B, Q, R, lo, hi = plant(rng, n, m)
        pb = (A, B, Q, R, Q, lo, hi)
    N = int(rng.integers(3, 8))
    dA, dB = rng.uniform(-e, e, (n * n, S)), rng.uniform(-e, e, (n * m, S))
    x0 = saturating_states(pb[0], pb[1], pb[2], pb[3], N, pb[5], pb[6], S, rng, t=t)
    return pb, dA, dB, x0, N


def _blk(M, s, r, c):
    return M[:, s].reshape(r, c)


def check_vs_oracle(pb, dA, dB, x0, N, h, rtol=1e-9):
    """Harness J and gradient against the oracle on every usable sample; returns (checked, with an active step)."""
    n, m = pb[1].shape
    done = act = 0
    for s in range(dA.shape[1]):
        if h["flags"][s] & ~FLAG_QP_ACTIVE or h["T_cert"][s] < 0:
            continue
        J, gA, gB, active = oracle_grad_inf(pb, _blk(dA, s, n, n), _blk(dB, s, n, m), x0[:, s], N, int(h["T_cert"][s]))
        assert abs(h["J"][s] - J) <= 1e-11 * abs(J), (s, h["J"][s], J)
        g = np.concatenate([gA.ravel(), gB.ravel()])
        hg = np.concatenate([h["gA"][:, s], h["gB"][:, s]])
        assert np.max(np.abs(hg - g)) <= rtol * np.max(np.abs(g)), (s, np.max(np.abs(hg - g)) / np.max(np.abs(g)))
        done += 1
        act += int(active > 0)
    return done, act


# ---------------------------------------------------------------------------------------------------- 1. gradient
@pytest.mark.parametrize("n,m", COMPILED_DIMS)
def test_gradient_vs_autograd(n, m):
    pb, dA, dB, x0, N = saturating_case(n, m, 700 + 10 * n + m)
    h = host_grad_inf(pb, dA, dB, x0, N)
    done, act = check_vs_oracle(pb, dA, dB, x0, N, h)
    assert done >= 3 and act == done, (done, act)


@pytest.mark.parametrize("n,m", [(2, 1), (3, 2), (4, 2), (3, 3)])
def test_gradient_general_weights_vs_autograd(n, m):
    pb, dA, dB, x0, N = saturating_case(n, m, 800 + 10 * n + m, general=True)
    h = host_grad_inf(pb, dA, dB, x0, N)
    done, act = check_vs_oracle(pb, dA, dB, x0, N, h)
    assert done >= 3 and act == done, (done, act)


def test_value_equals_simulate_inf():
    """J_inf, T_cert and flags of the gradient pass equal K2c's (the same header code computes them)."""
    for n, m in ((2, 1), (4, 2), (3, 3)):
        pb, dA, dB, x0, N = saturating_case(n, m, 900 + 10 * n + m, S=6)
        A, B, Q, R, _, lo, hi = pb
        J, Tc, fl = host_inf(A, B, Q, R, lo, hi, dA, dB, N, 1000, x0)
        for grad in (False, True):
            h = host_grad_inf(pb, dA, dB, x0, N, grad=grad)
            assert np.array_equal(h["J"], J) and np.array_equal(h["T_cert"], Tc) and np.array_equal(h["flags"], fl)


# ---------------------------------------------------------------------------------------------------- 2. reductions
@pytest.mark.parametrize("n,m", [(1, 1), (2, 1), (4, 2), (6, 2)])
def test_no_bounds_is_worst_eval(n, m):
    rng = np.random.default_rng(1000 + 10 * n + m)
    A, B, Q, R, _, _ = plant(rng, n, m)
    N, S = 6, 5
    dA, dB = rng.uniform(-0.01, 0.01, (n * n, S)), rng.uniform(-0.01, 0.01, (n * m, S))
    x0 = rng.normal(size=(n, S))
    h = host_grad_inf((A, B, Q, R, Q, None, None), dA, dB, x0, N)
    w = host_grad((A, B, Q, R, Q), dA, dB, x0, N)
    assert np.all(h["T_cert"] == 0) and np.array_equal(h["flags"], w["flags"])
    assert np.max(np.abs(h["J"] - w["J"]) / w["J"]) <= 1e-12
    for k in ("gA", "gB"):
        assert np.max(np.abs(h[k] - w[k])) <= 1e-12 * np.max(np.abs(w[k]))


def test_inside_the_certificate_is_the_unconstrained_gradient():
    """x0 small enough to start inside the certified set (tau = 0): the gradient of the unconstrained law's J."""
    for n, m in ((2, 1), (3, 2), (4, 2)):
        pb, dA, dB, x0, N = saturating_case(n, m, 1100 + 10 * n + m)
        x0 = x0 * 1e-3
        h = host_grad_inf(pb, dA, dB, x0, N)
        w = host_grad(pb[:5], dA, dB, x0, N)
        assert np.all(h["T_cert"] == 0) and not np.any(h["flags"])
        assert np.max(np.abs(h["J"] - w["J"]) / w["J"]) <= 1e-12
        for k in ("gA", "gB"):
            assert np.max(np.abs(h[k] - w[k])) <= 1e-12 * np.max(np.abs(w[k]))


def _along(pb, dA, dB, x0, N, d, ts):
    n, m = pb[1].shape
    S = len(ts)
    a = dA[:, :1] + d[:n * n, None] * ts[None, :]
    b = dB[:, :1] + d[n * n:, None] * ts[None, :]
    return host_grad_inf(pb, a, b, np.repeat(x0[:, :1], S, axis=1), N)


def test_tau_moves_continuously():
    """Along a line in (dA, dB) where the certified step changes by one, J changes by O(h) across the switch and the
    gradients on its two sides agree."""
    found = 0
    for seed in range(1200, 1230):
        pb, dA, dB, x0, N = saturating_case(2, 1, seed, S=1)
        rng = np.random.default_rng(seed)
        d = rng.normal(size=6)
        d /= np.linalg.norm(d)
        ts = np.linspace(-0.05, 0.05, 201)
        h = _along(pb, dA, dB, x0, N, d, ts)
        ok = (h["flags"] & ~FLAG_QP_ACTIVE) == 0
        jump = np.flatnonzero(ok[:-1] & ok[1:] & (np.abs(np.diff(h["T_cert"])) == 1))
        if not jump.size:
            continue
        lo_t, hi_t = ts[jump[0]], ts[jump[0] + 1]
        t_lo = int(h["T_cert"][jump[0]])
        for _ in range(60):                                      # bisect the switch
            mid = 0.5 * (lo_t + hi_t)
            if _along(pb, dA, dB, x0, N, d, np.array([mid]))["T_cert"][0] == t_lo:
                lo_t = mid
            else:
                hi_t = mid
        hh = 1e-7
        e = _along(pb, dA, dB, x0, N, d, np.array([lo_t - hh, lo_t, hi_t, hi_t + hh]))
        assert e["T_cert"][1] != e["T_cert"][2]
        assert abs(e["J"][2] - e["J"][1]) <= 1e-12 * e["J"][1] + 1e-6 * abs(e["J"][3] - e["J"][0])
        g1 = np.concatenate([e["gA"][:, 1], e["gB"][:, 1]])
        g2 = np.concatenate([e["gA"][:, 2], e["gB"][:, 2]])
        assert np.max(np.abs(g1 - g2)) <= 1e-6 * np.max(np.abs(g1))
        found += 1
        if found == 3:
            break
    assert found >= 1


def test_central_differences():
    """An oracle-independent check away from kinks: the gradient against central differences of the harness's J."""
    checked = 0
    for n, m in ((2, 1), (3, 2), (4, 2)):
        pb, dA, dB, x0, N = saturating_case(n, m, 1300 + 10 * n + m, S=3)
        h = host_grad_inf(pb, dA, dB, x0, N)
        for s in range(3):
            if h["flags"][s] != FLAG_QP_ACTIVE:
                continue
            g = np.concatenate([h["gA"][:, s], h["gB"][:, s]])
            base = np.concatenate([dA[:, s], dB[:, s]])
            E = 1e-6 * np.eye(len(base))
            pts = np.concatenate([base[:, None] + E, base[:, None] - E], axis=1)
            k = len(base)
            f = host_grad_inf(pb, pts[:n * n], pts[n * n:], np.repeat(x0[:, s:s + 1], 2 * k, axis=1), N, grad=False)
            fd = (f["J"][:k] - f["J"][k:]) / 2e-6
            assert np.max(np.abs(fd - g)) <= 1e-5 * np.max(np.abs(g)), (n, m, s)
            checked += 1
    assert checked >= 5


# ---------------------------------------------------------------------------------------------------- 3. ascent
def residual(pb, dA, dB, x0, N, eA, eB, norm):
    """r = ||Proj(u + g^/||g^||) - u||_2 in u = (dA/eA, dB/eB) with the harness gradient (one sample, matrices)."""
    n, m = pb[1].shape
    h = host_grad_inf(pb, dA.reshape(-1, 1), dB.reshape(-1, 1), x0.reshape(n, 1), N)
    gA, gB = h["gA"][:, 0].reshape(n, n), h["gB"][:, 0].reshape(n, m)
    gn = np.sqrt(eA ** 2 * np.sum(gA ** 2) + eB ** 2 * np.sum(gB ** 2))
    if gn == 0:
        return 0.0
    r2 = 0.0
    for M, g, e in ((dA, gA, eA), (dB, gB, eB)):
        if e > 0:
            r2 += np.sum((project(M + e * e * g / gn, e, norm) - M) ** 2) / e ** 2
    return float(np.sqrt(r2))


def ascent_cases():
    """(problem, dA, dB, x0, N, e_A, e_B) of the ascent checks: saturating 2 x 1 and 4 x 2 plants, one with an e = 0
    block."""
    out = []
    for (n, m, seed, eA, eB) in ((2, 1, 1400, 0.05, 0.05), (4, 2, 1401, 0.02, 0.0)):
        pb, dA, dB, x0, N = saturating_case(n, m, seed, S=5, e=eA)
        out.append((pb, dA, dB * (eB > 0), x0, N, eA, eB))
    return out


@pytest.mark.parametrize("norm", ["max", "f", "2"])
def test_ascent(norm):
    conv = 0
    for pb, dA, dB, x0, N, eA, eB in ascent_cases():
        n, m = pb[1].shape
        got = host_ascent_inf(pb, dA, dB, x0, N, eA, eB, norm)
        start = host_ascent_inf(pb, dA, dB, x0, N, eA, eB, norm, max_iter=0)
        for s in range(dA.shape[1]):
            a, b = _blk(got["dA"], s, n, n), _blk(got["dB"], s, n, m)
            assert feasible(a, eA, norm) and feasible(b, eB, norm), s
            if eB == 0:
                assert np.all(b == 0)
            assert got["J"][s] >= start["J"][s], s
            if got["flags"][s] & FLAG_UNSTABLE:
                assert np.isinf(got["J"][s])
                continue
            v = host_grad_inf(pb, a.reshape(-1, 1), b.reshape(-1, 1), x0[:, s:s + 1], N, grad=False)
            assert v["J"][0] == got["J"][s] and v["T_cert"][0] == got["T_cert"][s]
            if not got["flags"][s] & FLAG_ASCENT_MAXITER:
                assert not got["flags"][s] & ~FLAG_QP_ACTIVE
                assert residual(pb, a, b, x0[:, s], N, eA, eB, norm) <= 1e-8 + 1e-8, s
                conv += 1
    assert conv >= 4


@pytest.mark.parametrize("norm", ["max", "f", "2"])
def test_wide_box_is_the_unconstrained_ascent(norm):
    """A box that never binds: the ascent of K1's J (worst_ascent)."""
    rng = np.random.default_rng(1500)
    A, B, Q, R, _, _ = plant(rng, 3, 2)
    lo, hi = -1e6 * np.ones(2), 1e6 * np.ones(2)
    N, S, e = 6, 4, 0.03
    dA, dB, x0 = rng.uniform(-e, e, (9, S)), rng.uniform(-e, e, (6, S)), rng.normal(size=(3, S))
    got = host_ascent_inf((A, B, Q, R, Q, lo, hi), dA, dB, x0, N, e, e, norm)
    ref = host_ascent((A, B, Q, R, Q), dA, dB, x0, N, e, e, norm)
    assert np.all(got["T_cert"] == 0)
    assert np.array_equal(got["flags"], ref["flags"]) and np.array_equal(got["iters"], ref["iters"])
    assert np.max(np.abs(got["J"] - ref["J"]) / ref["J"]) <= 1e-12
    assert np.max(np.abs(got["dA"] - ref["dA"])) <= 1e-12 and np.max(np.abs(got["dB"] - ref["dB"])) <= 1e-12


def scalar_tight_box():
    A, B, Q, R = np.array([[1.1]]), np.array([[0.8]]), np.array([[1.0]]), np.array([[0.5]])
    return (A, B, Q, R, Q, np.array([-0.6]), np.array([0.6])), 3, 0.2, 1.3


def test_scalar_tight_box_matches_grid_search():
    """n = m = 1 with a box that binds on the first steps: the best ascent from a 5 x 5 grid of starts reaches a fine
    grid's maximum of K2c's J_inf, and that worst case is not the unconstrained law's."""
    pb, N, e, x0 = scalar_tight_box()
    g = np.linspace(-e, e, 201)
    a, b = np.repeat(g, len(g))[None, :], np.tile(g, len(g))[None, :]
    v = host_grad_inf(pb, a, b, np.full((1, a.shape[1]), x0), N, grad=False)
    assert np.all(v["flags"] & ~FLAG_QP_ACTIVE == 0)
    grid_max = v["J"].max()
    s = np.linspace(-e, e, 5)
    dA, dB = np.repeat(s, 5)[None, :], np.tile(s, 5)[None, :]
    got = host_ascent_inf(pb, dA, dB, np.full((1, 25), x0), N, e, e, "max")
    assert not np.any(got["flags"] & ~FLAG_QP_ACTIVE)
    assert got["J"].max() >= grid_max * (1 - 1e-9)
    unc = host_ascent(pb[:5], dA, dB, np.full((1, 25), x0), N, e, e, "max")
    i, j = int(np.argmax(got["J"])), int(np.argmax(unc["J"]))
    assert abs(got["J"][i] - unc["J"][j]) > 1e-3 * unc["J"][j]
    assert abs(got["dA"][0, i] - unc["dA"][0, j]) + abs(got["dB"][0, i] - unc["dB"][0, j]) > 1e-3


def test_ascent_finds_a_destabilising_error():
    A, B, Q, R = np.array([[1.3, 0.2], [0.0, 0.9]]), np.array([[1.0], [0.3]]), np.eye(2), np.eye(1)
    pb, N, e = (A, B, Q, R, Q, np.array([-2.0]), np.array([2.0])), 8, 0.35
    rng = np.random.default_rng(2)
    dA, dB = rng.uniform(-0.02, 0.02, (4, 8)), rng.uniform(-0.02, 0.02, (2, 8))
    x0 = rng.normal(size=(2, 8))
    assert not np.any(host_grad_inf(pb, dA, dB, x0, N)["flags"] & ~FLAG_QP_ACTIVE)
    for norm in ("max", "f"):
        got = host_ascent_inf(pb, dA, dB, x0, N, e, e, norm)
        hit = np.flatnonzero(got["flags"] & FLAG_UNSTABLE)
        assert len(hit) >= 1
        for s in hit:
            assert np.isinf(got["J"][s]) and got["T_cert"][s] == -1 and got["rho"][s] >= 1
            assert feasible(_blk(got["dA"], s, 2, 2), e, norm) and feasible(_blk(got["dB"], s, 2, 1), e, norm)


def _nan_grad(h, s):
    return np.all(np.isnan(h["gA"][:, s])) and np.all(np.isnan(h["gB"][:, s]))


def test_failure_values():
    """UNSTABLE: J = +inf; TAIL_UNCERTIFIED: J = NaN, T_cert = -1; QP_MAXITER (N m > 256): K2c's J of the clipped
    inputs. The gradient is NaN in each, and the ascent returns such a start as it is."""
    # unstable: the model's input acts the other way
    pb = (np.array([[1.2]]), np.array([[1.0]]), np.eye(1), np.eye(1), np.eye(1), np.array([-1.0]), np.array([1.0]))
    z, one = np.zeros((1, 1)), np.ones((1, 1))
    h = host_grad_inf(pb, z, np.array([[-2.0]]), one, 5, 100)
    assert h["J"][0] == np.inf and h["T_cert"][0] == -1 and h["flags"][0] & FLAG_UNSTABLE and _nan_grad(h, 0)
    # budget below tau
    pbc, dA, dB, x0, N = saturating_case(4, 2, 1600, S=4)
    h = host_grad_inf(pbc, dA, dB, x0, N)
    s = int(np.argmax(h["T_cert"]))
    assert h["T_cert"][s] >= 2
    args = (pbc, dA[:, s:s + 1], dB[:, s:s + 1], x0[:, s:s + 1], N)
    u = host_grad_inf(*args, T_max=int(h["T_cert"][s]) - 1)
    assert np.isnan(u["J"][0]) and u["T_cert"][0] == -1 and u["flags"][0] & FLAG_TAIL_UNCERTIFIED and _nan_grad(u, 0)
    a = host_ascent_inf(*args, 0.05, 0.05, "max", T_max=int(h["T_cert"][s]) - 1)     # the start lies in the set
    assert a["iters"][0] == 0 and np.isnan(a["J"][0]) and a["flags"][0] & FLAG_TAIL_UNCERTIFIED
    assert np.array_equal(a["dA"], args[1]) and np.array_equal(a["dB"], args[2])
    # beyond the working-set mask: N m = 257
    pbm = (np.array([[0.9]]), np.array([[1.0]]), np.eye(1), np.eye(1), np.eye(1), np.array([-0.1]), np.array([0.1]))
    q = host_grad_inf(pbm, z, z, np.array([[50.0]]), 257)
    J, Tc, fl = host_inf(*pbm[:4], pbm[5], pbm[6], z, z, 257, 1000, np.array([[50.0]]))
    assert q["J"][0] == J[0] and q["flags"][0] == fl[0] and fl[0] & FLAG_QP_MAXITER and _nan_grad(q, 0)
    a = host_ascent_inf(pbm, z + 0.01, z, np.array([[50.0]]), 257, 0.05, 0.05, "max")
    assert a["iters"][0] == 0 and a["flags"][0] & FLAG_QP_MAXITER and a["dA"][0, 0] == 0.01
