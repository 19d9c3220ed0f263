"""K1's closed-loop cost from the characteristic polynomial of A_cl (riccati.cuh: lyapunov_cost_poly, n = 3, 4).

J = x0' S x0 with S = W + A_cl' S A_cl is taken from a Cayley-Hamilton linear system where that route accepts its own
result, and from the Lyapunov doubling everywhere else. CPU tier: the g++ build of the same header against a 50-digit
Stein solve on closed loops that are easy, clustered, defective, nilpotent, near the stability boundary or strongly
non-normal, and on the closed loops of the synthetic problem. GPU tier: K1 against that host build, and the default
build against LQMPC_K1_LYAP=doubling."""
import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile

import mpmath as mp
import numpy as np
import pytest

from oracle import np_batched as nb
from tests.hostmath import api as hm

N_HOR = 10
_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def _cost_lib():
    """g++ build of tests/k1_closed_loop_cost_host.cpp (riccati.cuh's routines), in a temporary directory."""
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="k1_cost_host_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libk1cost.so")
        r = subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-x", "c++",
                            os.path.join(_HERE, "k1_closed_loop_cost_host.cpp"), "-o", so, "-lm"],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        _lib = ctypes.CDLL(so)
    return _lib


def closed_loop_cost(Acl, W, x0):
    """x0' S x0 of S = W + Acl' S Acl (n = 3, 4; AoS operands [S, n, n], [S, n, n], [S, n]) by K1's
    characteristic-polynomial route and by the Lyapunov doubling: (J_poly, accepted, J_doubling, doubling_converged).
    J_poly is NaN where the polynomial route was not reached (rho >= 1 or the closed-form spectrum was not trusted)."""
    c = [np.ascontiguousarray(a, dtype=np.float64) for a in (Acl, W, x0)]
    S, n = c[0].shape[0], c[0].shape[1]
    assert c[1].shape == (S, n, n) and c[2].shape == (S, n)
    Jp, Jd = np.zeros(S), np.zeros(S)
    acc, dok = np.zeros(S, dtype=np.int32), np.zeros(S, dtype=np.int32)
    P, I32 = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int32)
    rc = _cost_lib().k1_closed_loop_cost(n, ctypes.c_int64(S), *[a.ctypes.data_as(P) for a in c],
                                         Jp.ctypes.data_as(P), acc.ctypes.data_as(I32), Jd.ctypes.data_as(P),
                                         dok.ctypes.data_as(I32))
    assert rc == 0
    return Jp, acc == 1, Jd, dok == 1


def stein_cost_truth(Acl, W, x0):
    """x0' S x0 with S = W + Acl' S Acl, by a 50-digit solve of the Stein equation in its symmetric vec form (the
    n (n + 1) / 2 entries S_ij, i <= j) from the given float64 Acl, W, x0."""
    with mp.workdps(50):
        A = mp.matrix(np.asarray(Acl, dtype=float).tolist())
        Wm = mp.matrix(np.asarray(W, dtype=float).tolist())
        n = A.rows
        x = [mp.mpf(float(v)) for v in np.asarray(x0, dtype=float).reshape(-1)]
        idx = [(i, j) for i in range(n) for j in range(i, n)]
        pos = {p: k for k, p in enumerate(idx)}
        big = mp.eye(len(idx))
        for r, (i, j) in enumerate(idx):          # S_ij - sum_kl A_ki A_lj S_kl = W_ij
            for k in range(n):
                for l in range(n):
                    big[r, pos[(k, l) if k <= l else (l, k)]] -= A[k, i] * A[l, j]
        vs = mp.lu_solve(big, mp.matrix([Wm[i, j] for (i, j) in idx]))
        J = mp.mpf(0)
        for (i, j), k in pos.items():
            J += (1 if i == j else 2) * x[i] * x[j] * vs[k]
        return float(J)


def _with_rho(M, rho):
    return M * (rho / np.max(np.abs(np.linalg.eigvals(M)), axis=1))[:, None, None]


def _similar(rng, D, cond_scale):
    """V D V^-1 with V = U diag(s) U', s log-uniform over cond_scale decades."""
    S, n, _ = D.shape
    U, _ = np.linalg.qr(rng.normal(size=(S, n, n)))
    s = 10.0 ** rng.uniform(0.0, cond_scale, size=(S, n))
    V = U * s[:, None, :] @ U.transpose(0, 2, 1)
    return V @ D @ np.linalg.inv(V)


def _families(n, S, seed):
    rng = np.random.default_rng(seed)
    g = rng.normal(size=(S, n, n))
    out = {
        "gauss": _with_rho(g, rng.uniform(0.05, 0.95, size=S)),
        "scaled": _with_rho(np.exp(rng.uniform(-3, 3, size=(S, n, 1))) * rng.normal(size=(S, n, n)) *
                            np.exp(rng.uniform(-3, 3, size=(S, 1, n))), rng.uniform(0.05, 0.95, size=S)),
        "clustered": 0.8 * np.eye(n)[None] + 0.02 * rng.normal(size=(S, n, n)),
        "tight": 0.9 * np.eye(n)[None] + 1e-3 * rng.normal(size=(S, n, n)),
        "near_unit": _with_rho(rng.normal(size=(S, n, n)), rng.uniform(0.9, 0.999, size=S)),
    }
    lam = rng.uniform(-0.9, 0.9, size=(S, 1, 1))
    out["defective"] = _similar(rng, lam * np.eye(n)[None] + np.eye(n, k=1)[None] * rng.uniform(0.1, 1.0, (S, 1, 1)), 1)
    out["nilpotent"] = _similar(rng, np.triu(rng.normal(size=(S, n, n)), 1), 1)
    d = rng.uniform(-0.95, 0.95, size=(S, n))
    out["non_normal"] = _similar(rng, d[:, :, None] * np.eye(n)[None], 4)
    fams = {}
    for k, A in out.items():
        L = rng.normal(size=(S, n, n))
        W = L @ L.transpose(0, 2, 1) + 1e-3 * np.eye(n)[None]
        fams[k] = (A, W, rng.normal(size=(S, n)))
    return fams


def _synth_closed_loops(n, m, S, e, seed):
    """A_cl = A + B K and W = Q + K' R K of K1's horizon-10 gain on the synthetic problem, perturbation level e."""
    A, B, Q, R = nb.synth_problem(n, m, seed=0)
    dA, dB, x0 = nb.synth_samples(n, m, S, seed=seed, e=e)
    got = hm.eval_batch(A, B, Q, R, Q, 30, *nb.to_soa(dA, dB, x0), N_HOR, N_HOR, 0)
    K = got["K0"][0].T.reshape(S, m, n)
    return A[None] + B[None] @ K, Q[None] + K.transpose(0, 2, 1) @ R[None] @ K, x0


def _check_family(name, Acl, W, x0, n_truth=60):
    Jp, acc, Jd, _ = closed_loop_cost(Acl, W, x0)
    rho = np.max(np.abs(np.linalg.eigvals(Acl)), axis=1)
    assert not np.any(acc & ~(rho < 1.0)), name
    # the accepted results that disagree most with the doubling, plus a random draw, against the 50-digit solve
    rel = np.where(acc, np.abs(Jp - Jd) / np.abs(Jd), -1.0)
    order = np.argsort(-rel)
    pick = set(order[:n_truth // 2][rel[order[:n_truth // 2]] >= 0].tolist())
    pick |= set(np.random.default_rng(1).choice(np.flatnonzero(acc), size=min(n_truth // 2, int(acc.sum())),
                                                 replace=False).tolist()) if acc.any() else set()
    for s in sorted(pick):
        t = stein_cost_truth(Acl[s], W[s], x0[s])
        assert abs(Jp[s] - t) <= 1e-11 * abs(t), (name, s, Jp[s], t, rho[s])
    return acc, rho


@pytest.mark.parametrize("n", [3, 4])
def test_accepted_cost_matches_50_digit_stein_solve(n):
    for name, (Acl, W, x0) in _families(n, 4000, 20 + n).items():
        acc, rho = _check_family(name, Acl, W, x0)
        if name == "gauss":
            assert acc[rho < 0.9].mean() > 0.999, (name, acc.mean())


@pytest.mark.parametrize("e", [0.01, 0.3, 0.6])
def test_synthetic_closed_loops(e):
    Acl, W, x0 = _synth_closed_loops(4, 2, 4000, e, seed=7)
    acc, _ = _check_family("synth e=%g" % e, Acl, W, x0)
    if e == 0.01:
        assert acc.mean() >= 0.999, acc.mean()


def test_headline_distribution_is_accepted():
    """The closed loops bench.py's headline draws (synthetic 4 x 2, e = 0.01, horizon 10) take the fast route."""
    Acl, W, x0 = _synth_closed_loops(4, 2, 20000, 0.01, seed=1)
    Jp, acc, Jd, _ = closed_loop_cost(Acl, W, x0)
    assert acc.mean() >= 0.999, acc.mean()
    assert np.max(np.abs(Jp[acc] - Jd[acc]) / Jd[acc]) < 1e-13


@pytest.mark.parametrize("n,m,e", [(4, 2, 0.01), (4, 2, 0.6), (3, 2, 0.3), (4, 1, 0.05)])
def test_eval_falls_back_to_doubling(n, m, e):
    """eval_sample: a sample the polynomial route does not accept gets the doubling's J and its flags. (A_cl and W are
    rebuilt here in numpy, so they differ from the kernel's in the last bits.)"""
    A, B, Q, R = nb.synth_problem(n, m, seed=0)
    S = 2000
    dA, dB, x0 = nb.synth_samples(n, m, S, seed=3, e=e)
    got = hm.eval_batch(A, B, Q, R, Q, 30, *nb.to_soa(dA, dB, x0), N_HOR, N_HOR, 0)
    K = got["K0"][0].T.reshape(S, m, n)
    Acl, W = A[None] + B[None] @ K, Q[None] + K.transpose(0, 2, 1) @ R[None] @ K
    Jp, acc, Jd, dok = closed_loop_cost(Acl, W, x0)
    J = got["J"][0]
    stable = (got["flags"][0] & 1) == 0
    assert np.max(np.abs(J[acc] - Jp[acc]) / Jp[acc], initial=0.0) < 1e-12
    rej = stable & ~acc
    assert np.max(np.abs(J[rej] - Jd[rej]) / Jd[rej], initial=0.0) < 1e-12
    lyap_flag = (got["flags"][0] & 64) != 0
    assert np.array_equal(lyap_flag, stable & ~acc & ~dok)


GPU_CASES = [(4, 2, 0.01), (4, 2, 0.6), (3, 2, 0.3), (3, 3, 0.1), (4, 4, 0.2), (4, 1, 0.05), (3, 1, 0.1)]


def _gpu_runs(engine, monkeypatch, n, m, e, S=4096):
    A, B, Q, R = nb.synth_problem(n, m, seed=0)
    engine.set_problem(A, B, Q, R, Q, None, None, 30)
    dA, dB, x0 = nb.synth_samples(n, m, S, seed=11, e=e)
    soa = nb.to_soa(dA, dB, x0)
    out = {}
    for mode in ("poly", "doubling"):
        if mode == "doubling":
            monkeypatch.setenv("LQMPC_K1_LYAP", "doubling")
        else:
            monkeypatch.delenv("LQMPC_K1_LYAP", raising=False)
        for hor in ((N_HOR, N_HOR), (2, 11)):
            g = engine.eval_batch(*soa, *hor)
            out[mode, hor] = {k: g[k].cpu().numpy() for k in ("J", "rho", "flags")}
        sd = engine.eval_seeded(5, 0, S, e, e, N_HOR, N_HOR, want=("J", "rho", "flags"))
        out[mode, "seeded"] = {k: sd[k].cpu().numpy() for k in ("J", "rho", "flags")}
    monkeypatch.delenv("LQMPC_K1_LYAP", raising=False)
    host = {hor: hm.eval_batch(A, B, Q, R, Q, 30, *soa, *hor, 0) for hor in ((N_HOR, N_HOR), (2, 11))}
    return out, host


def _rel(a, b):
    return np.abs(a - b) / np.maximum(np.abs(b), 1e-300)


def _host_device_tol(rho):
    """Allowance between two J of the same closed loop computed along different rounding paths: the host and device
    builds (FMA contraction, reciprocals: A_cl differs in the last bits) or the two closed-loop routes. Up to rho = 0.9
    that moves J by < 1e-13; nearer the boundary J's condition grows like rho / (1 - rho), and two results that are each
    within 1e-11 of the 50-digit value may differ by twice that."""
    u = 2.0 ** -53
    return np.where(rho <= 0.9, 1e-12, np.maximum(2e-11, 64 * u * rho / np.maximum(1.0 - rho, 1e-300)))


@pytest.mark.gpu
@pytest.mark.parametrize("n,m,e", GPU_CASES)
def test_gpu_k1_matches_host_build_and_doubling_build(engine, monkeypatch, n, m, e):
    out, host = _gpu_runs(engine, monkeypatch, n, m, e)
    for hor in ((N_HOR, N_HOR), (2, 11)):
        g, h = out["poly", hor], host[hor]
        well = np.abs(h["rho"] - 1.0) > 1e-6
        fin = well & np.isfinite(h["J"])
        assert np.array_equal(np.isfinite(g["J"][well]), np.isfinite(h["J"][well])), hor
        assert np.all(_rel(g["J"][fin], h["J"][fin]) <= _host_device_tol(h["rho"][fin])), hor
        assert np.max(_rel(g["rho"][well], h["rho"][well]), initial=0.0) < 1e-12, hor
        assert np.array_equal(g["flags"][well], h["flags"][well]), hor
    for key in ((N_HOR, N_HOR), (2, 11), "seeded"):
        p, d = out["poly", key], out["doubling", key]
        assert np.array_equal(p["rho"], d["rho"]), key                # the spectrum is computed exactly as before
        assert np.array_equal(p["flags"] & ~64, d["flags"] & ~64), key
        fin = np.isfinite(d["J"])
        assert np.array_equal(np.isfinite(p["J"]), fin), key
        assert np.all(_rel(p["J"][fin], d["J"][fin]) <= _host_device_tol(d["rho"][fin])), key
