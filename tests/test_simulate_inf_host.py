"""CPU tier — the infinite-horizon closed loop of K2c (clqr.cuh: simulate_inf_sample / inf_tail; pclqr.cuh:
psimulate_inf_sample / poly_certificate) compiled with g++ from the engine headers (tests/hostmath/inf.cpp, the flags
of tests/hostmath/build.py), against a numpy oracle of the same method built on np_oracle.mpc_solve and
scipy.linalg.solve_discrete_lyapunov. The GPU tier (tests/test_simulate_inf.py) runs the device kernels against this
harness and the oracle."""
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import pytest
import scipy.linalg as sla

from oracle import np_oracle as o
from tests.conftest import random_polytope

HERE = os.path.dirname(os.path.abspath(__file__))
HM = os.path.join(HERE, "hostmath")
CSRC = os.path.join(os.path.dirname(HERE), "lq_mpc_b200", "csrc")
COMPILED_DIMS = [(1, 1), (2, 1), (2, 2), (3, 1), (3, 2), (3, 3), (4, 1), (4, 2), (4, 4), (6, 2), (8, 2)]
TOL = 1e-9
FLAG_UNSTABLE, FLAG_TAIL_UNCERTIFIED = 1, 1024

_P = ctypes.POINTER(ctypes.c_double)
_I = ctypes.POINTER(ctypes.c_int32)
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(HM, "_build")
        os.makedirs(out, exist_ok=True)
        so = os.path.join(out, "libinf.so")
        src = os.path.join(HM, "inf.cpp")
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


def host_inf(A, B, Q, R, lo, hi, dA, dB, N, T_max, x0, F=None):
    """Harness K2c: J_inf [S], T_cert [S], flags [S] (dA [n*n][S], dB [n*m][S], x0 [n][S]; F: polytope rows)."""
    n, m = B.shape
    S = dA.shape[1]
    keep = [_c(a) for a in (A, B, Q, R, Q, lo, hi, dA, dB, x0, F)]
    J, Tc, fl = np.zeros(S), np.zeros(S, dtype=np.int32), np.zeros(S, dtype=np.int32)
    rc = lib().inf_sim(n, m, *[_p(a) for a in keep[:7]], ctypes.c_int64(S), _p(keep[7]), _p(keep[8]), N, T_max,
                       _p(keep[9]), _p(keep[10]), 0 if F is None else F.shape[0], _p(J), Tc.ctypes.data_as(_I),
                       fl.ctypes.data_as(_I))
    assert rc == 0
    return J, Tc, fl


def host_tail(A, B, Q, R, lo, hi, Ah, Bh, N, F=None):
    """Harness certificate of one model: (S, c_S, cstar, gains K [N][m][n], flags)."""
    n, m = B.shape
    keep = [_c(a) for a in (A, B, Q, R, Q, lo, hi, (Ah - A).reshape(-1), (Bh - B).reshape(-1), F)]
    S, cS, cs, K = np.zeros(n * n), np.zeros(1), np.zeros(1), np.zeros(N * m * n)
    f = lib().inf_tail(n, m, *[_p(a) for a in keep[:9]], N, _p(keep[9]), 0 if F is None else F.shape[0], _p(S),
                       _p(cS), _p(cs), _p(K))
    assert f >= 0
    return S.reshape(n, n), float(cS[0]), float(cs[0]), K.reshape(N, m, n), f


def oracle_inf(A, B, Ah, Bh, Q, R, lo, hi, x0, N, T_max=1000, F=None):
    """The method in numpy: (J_inf, tau); tau = -2 unstable (J = inf), -1 not certified within T_max (J = NaN)."""
    n, m = Bh.shape
    K, P = o.riccati(Ah, Bh, Q, R, Q, N)
    P0i = np.linalg.inv(P[0])
    cs, Phi = np.inf, np.eye(n)
    for k in range(N):
        g = K[k] @ Phi
        rows = [(f @ g, 1.0) for f in F] if F is not None else \
            [(g[j], min(-lo[j], hi[j]) ** 2) for j in range(m)] if lo is not None else []
        for h, b2 in rows:
            q = h @ P0i @ h
            if q > 0:
                cs = min(cs, b2 / q)
        Phi = (Ah + Bh @ K[k]) @ Phi
    cs *= 1 - 1e-9
    Acl, W = A + B @ K[0], Q + K[0].T @ R @ K[0]
    if not o.spectral_radius(Acl) < 1:
        return np.inf, -2
    S = sla.solve_discrete_lyapunov(Acl.T, W)
    Li = np.linalg.inv(np.linalg.cholesky(S))
    cS = (1 - 1e-9) * cs / np.max(np.linalg.eigvalsh(Li @ P[0] @ Li.T))
    x, cost = np.array(x0, dtype=float), 0.0
    for t in range(T_max + 1):
        if x @ S @ x <= cS:
            return cost + x @ S @ x, t
        if t == T_max:
            return np.nan, -1
        u, _, _ = o.mpc_solve(N, Ah, Bh, Q, R, Q, lo, hi, x, True, (K, P), F_u=F)
        cost += x @ Q @ x + u @ R @ u
        x = A @ x + B @ u


def plant(rng, n, m):
    A = rng.normal(size=(n, n)); A *= rng.uniform(0.8, 1.05) / o.spectral_radius(A)
    B = rng.normal(size=(n, m))
    Q, R = rng.uniform(0.5, 3) * np.eye(n), rng.uniform(0.1, 2) * np.eye(m)
    lo, hi = -rng.uniform(0.1, 0.4, size=m), rng.uniform(0.1, 0.4, size=m)
    return A, B, Q, R, lo, hi


def saturating_states(A, B, Q, R, N, lo, hi, S, rng, F=None, t=(1.5, 4.0)):
    """[n][S] states whose unconstrained nominal plan peaks at t times the input set (linear in the state)."""
    n, m = B.shape
    K, _ = o.riccati(A, B, Q, R, Q, N)
    x0 = rng.normal(size=(n, S))
    x, r = x0.copy(), np.zeros(S)
    for k in range(N):
        u = K[k] @ x
        r = np.maximum(r, np.max(F @ u, axis=0) if F is not None else np.maximum(u / hi[:, None], u / lo[:, None]).max(0))
        x = A @ x + B @ u
    return x0 * rng.uniform(*t, size=S) / r


def case(n, m, seed, S=6, poly=False):
    rng = np.random.default_rng(seed)
    A, B, Q, R, lo, hi = plant(rng, n, m)
    N = int(rng.integers(3, 10))
    F = random_polytope(rng, m, 2 * m + 1, 0.15, 0.45) if poly else None
    if poly:
        lo = hi = None
    dA = rng.uniform(-0.01, 0.01, size=(n * n, S)); dB = rng.uniform(-0.01, 0.01, size=(n * m, S))
    x0 = saturating_states(A, B, Q, R, N, lo, hi, S, rng, F)
    return dict(A=A, B=B, Q=Q, R=R, lo=lo, hi=hi, F=F, N=N, dA=dA, dB=dB, x0=x0)


def model(c, s):
    n, m = c["B"].shape
    return c["A"] + c["dA"][:, s].reshape(n, n), c["B"] + c["dB"][:, s].reshape(n, m)


def check_vs_oracle(c, J, Tc, fl, T_max=1000):
    certified = 0
    for s in range(c["dA"].shape[1]):
        Ah, Bh = model(c, s)
        Jo, to = oracle_inf(c["A"], c["B"], Ah, Bh, c["Q"], c["R"], c["lo"], c["hi"], c["x0"][:, s], c["N"], T_max,
                            c["F"])
        if to == -2:
            assert J[s] == np.inf and Tc[s] == -1 and fl[s] & FLAG_UNSTABLE, s
        elif to == -1:
            assert np.isnan(J[s]) and Tc[s] == -1 and fl[s] & FLAG_TAIL_UNCERTIFIED, s
        else:
            assert abs(J[s] - Jo) <= TOL * Jo, (s, J[s], Jo)
            assert Tc[s] >= 0 and abs(int(Tc[s]) - to) <= 1, (s, Tc[s], to)   # (c_S rounding at the boundary)
            assert not fl[s] & (FLAG_UNSTABLE | FLAG_TAIL_UNCERTIFIED)
            certified += 1
    return certified


@pytest.mark.parametrize("n,m", COMPILED_DIMS)
def test_box_matches_oracle_every_pair(n, m):
    c = case(n, m, 100 + 10 * n + m)
    J, Tc, fl = host_inf(c["A"], c["B"], c["Q"], c["R"], c["lo"], c["hi"], c["dA"], c["dB"], c["N"], 1000, c["x0"])
    assert check_vs_oracle(c, J, Tc, fl) >= 3
    assert np.any(fl & 2), "no step with an active bound: the case does not exercise the constrained steps"


@pytest.mark.parametrize("n,m", [d for d in COMPILED_DIMS if d[1] >= 2])
def test_polytope_matches_oracle(n, m):
    c = case(n, m, 200 + 10 * n + m, S=4, poly=True)
    J, Tc, fl = host_inf(c["A"], c["B"], c["Q"], c["R"], None, None, c["dA"], c["dB"], c["N"], 1000, c["x0"], c["F"])
    assert check_vs_oracle(c, J, Tc, fl) >= 2
    assert np.any(fl & 2)


@pytest.mark.parametrize("n,m", [(2, 1), (4, 2), (3, 3)])
def test_identity_with_finite_horizon_cost(n, m):
    """J_inf = J_T(T) + x_T'(S - Q) x_T for every T >= tau (J_T, x_T from np_oracle.simulate)."""
    c = case(n, m, 300 + 10 * n + m, S=4)
    J, Tc, fl = host_inf(c["A"], c["B"], c["Q"], c["R"], c["lo"], c["hi"], c["dA"], c["dB"], c["N"], 1000, c["x0"])
    done = 0
    for s in np.flatnonzero(Tc >= 0):
        Ah, Bh = model(c, s)
        S = host_tail(c["A"], c["B"], c["Q"], c["R"], c["lo"], c["hi"], Ah, Bh, c["N"])[0]
        for T in (int(Tc[s]), int(Tc[s]) + 7):
            sim = o.simulate(T, c["N"], Ah, Bh, c["Q"], c["R"], c["Q"], c["lo"], c["hi"], c["x0"][:, s], c["A"], c["B"])
            xT = sim["X"][:, T]
            assert abs(sim["J_T"] + xT @ (S - c["Q"]) @ xT - J[s]) <= TOL * J[s]
        done += 1
    assert done >= 2


def test_golden_inputs_certified_and_equal_to_shipped_cost(golden, example):
    """All 1 500 evaluations of the shipped sweep: certified by step 30, and J_inf equals the shipped J_T(30) (the tail
    beyond 30 steps is ~1e-35 at spectral radii 0.18-0.26)."""
    z, ex = golden, example
    A, B, Q, R, lo, hi = ex["A"], ex["B"], ex["Q"], ex["R"], ex["lo"], ex["hi"]
    xs = o.circle_generator(8, 1.5, o.local_radius(lo, hi, -o.dlqr(A, B, Q, R)[0], Q), Q)[:, 1]
    eA, eB = z["error_A_f"], z["error_B_f"]
    cells = [(i, 7, z["true_cost_error"][:, i]) for i in range(eA.shape[3])] + \
        [(4, int(N), z["true_cost_horizon"][:, h]) for h, N in enumerate(z["horizon"])]
    assert sum(len(col) for _, _, col in cells) == 1500
    for i, N, col in cells:
        S = eA.shape[2]
        J, Tc, fl = host_inf(A, B, Q, R, lo, hi, eA[:, :, :, i].reshape(4, S), eB[:, :, :, i].reshape(2, S), N, 1000,
                             np.repeat(xs[:, None], S, axis=1))
        assert np.all((Tc >= 0) & (Tc <= 30)) and not np.any(fl & ~2)
        assert np.max(np.abs(J - col) / col) <= 1e-12


@pytest.mark.parametrize("n,m", [(1, 1), (2, 1), (4, 2), (6, 2)])
def test_no_bounds_is_the_unconstrained_cost(n, m):
    rng = np.random.default_rng(400 + 10 * n + m)
    A, B, Q, R, _, _ = plant(rng, n, m)
    N, S = 6, 5
    dA = rng.uniform(-0.01, 0.01, size=(n * n, S)); dB = rng.uniform(-0.01, 0.01, size=(n * m, S))
    x0 = rng.normal(size=(n, S))
    J, Tc, fl = host_inf(A, B, Q, R, None, None, dA, dB, N, 0, x0)
    assert np.all(Tc == 0) and not np.any(fl)
    for s in range(S):
        Ah, Bh = A + dA[:, s].reshape(n, n), B + dB[:, s].reshape(n, m)
        Jo, _ = o.closed_loop_inf_cost(A, B, o.riccati(Ah, Bh, Q, R, Q, N)[0][0], Q, R, x0[:, s])
        assert abs(J[s] - Jo) <= 1e-11 * Jo


def test_unstable_true_closed_loop_is_infinite():
    A, B, Q, R = np.array([[1.2]]), np.array([[1.0]]), np.eye(1), np.eye(1)
    dB = np.array([[-2.0]])                                 # the model's input acts the other way: A + B K0 > 1.2
    J, Tc, fl = host_inf(A, B, Q, R, np.array([-1.0]), np.array([1.0]), np.zeros((1, 1)), dB, 5, 100, np.ones((1, 1)))
    assert J[0] == np.inf and Tc[0] == -1 and fl[0] & FLAG_UNSTABLE


def test_budget_below_tau_is_uncertified():
    c = case(4, 2, 501, S=6)
    args = (c["A"], c["B"], c["Q"], c["R"], c["lo"], c["hi"], c["dA"], c["dB"], c["N"])
    J, Tc, fl = host_inf(*args, 1000, c["x0"])
    late = np.flatnonzero(Tc >= 2)
    assert late.size
    s = late[0]
    J2, Tc2, fl2 = host_inf(*args, int(Tc[s]) - 1, c["x0"])
    assert np.isnan(J2[s]) and Tc2[s] == -1 and fl2[s] & FLAG_TAIL_UNCERTIFIED
    J3, Tc3, _ = host_inf(*args, int(Tc[s]), c["x0"])
    assert J3[s] == J[s] and Tc3[s] == Tc[s]


def _inside(F, lo, hi, u):
    if F is not None:
        return np.max(F @ u) <= 1.0 + 1e-12
    return np.all(u >= lo * (1 + 1e-12)) and np.all(u <= hi * (1 + 1e-12))


@pytest.mark.parametrize("n,m,poly", [(2, 1, False), (4, 2, False), (3, 3, False), (4, 2, True), (3, 3, True)])
def test_certificate_is_sound(n, m, poly):
    """From points on the boundary x'Sx = c_S the unconstrained plan stays inside the input set, and so does every plan
    along 50 further steps of the true closed loop under u = K0 x."""
    c = case(n, m, 600 + 10 * n + m, S=3, poly=poly)
    rng = np.random.default_rng(7)
    checked = 0
    for s in range(3):
        Ah, Bh = model(c, s)
        S, cS, cstar, K, f = host_tail(c["A"], c["B"], c["Q"], c["R"], c["lo"], c["hi"], Ah, Bh, c["N"], c["F"])
        if not (cS > 0):
            continue
        assert cstar > 0 and not f & FLAG_UNSTABLE
        Lt = np.linalg.cholesky(S).T
        Acl = c["A"] + c["B"] @ K[0]
        for _ in range(100):
            z = rng.normal(size=n)
            x = np.linalg.solve(Lt, z / np.linalg.norm(z)) * np.sqrt(cS)     # x'Sx = c_S
            for _t in range(51):
                xp = x
                for k in range(c["N"]):
                    u = K[k] @ xp
                    assert _inside(c["F"], c["lo"], c["hi"], u)
                    xp = Ah @ xp + Bh @ u
                assert x @ S @ x <= cS * (1 + 1e-12)
                x = Acl @ x
        checked += 1
    assert checked >= 2
