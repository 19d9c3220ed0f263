"""Shared inputs and checks of the K3 extended-precision tests (tests/test_bounds_truth.py on the GPU,
tests/test_bounds_truth_host.py on the g++ build of the same headers). Test infrastructure only.

Tolerances (relative, against tests/mp_truth.py at 50 digits):
  GRAM_TOL       matrix-free lambda_min(H^) and lambda_max(Gamma'Gamma): the bisection stops at a relative bracket
                 of 2^-42 = 2.3e-13 and each probe's answer is exact up to a backward error of a few ulps of the
                 probed matrix, so 1e-11 leaves a margin of 40;
  FIELD_TOL      every other field, times its condition factor 1 + kappa (mp_truth.k3_truth);
  EDGE_MARGIN    a sample whose decisive edge argument lies within this relative distance of the edge may carry
                 either flag value.
"""
from __future__ import annotations

import concurrent.futures as cf
import multiprocessing
import os
import zlib

import mpmath as mp
import numpy as np

from tests import mp_truth as mt

GRAM_TOL = 1e-11
FIELD_TOL = 1e-9
EDGE_MARGIN = 1e-9
U = 2.0 ** -53
SWEEP_A = np.array([[1.0, 0.7], [0.12, 0.4]])          # cfg-sweep-f's plant: rho(A) = 1.117, open-loop unstable
SWEEP_B = np.array([[1.0], [1.2]])
SWEEP_Q, SWEEP_R = 2.0 * np.eye(2), np.eye(1)
SWEEP_LO, SWEEP_HI = np.array([-0.1]), np.array([0.1])
P3 = np.array([0.1, 1.0, 0.6])
SWEEP_ERRORS = np.linspace(1e-3, 1e-2, 10)
GRAM_HORIZONS = (1, 2, 12, 13, 30, 50)


def pmap(fn, args):
    """fn(*a) for a in args on every CPU (spawned workers: safe after CUDA is initialised)."""
    args = list(args)
    workers = min(len(args), os.cpu_count() or 1, 32)
    if workers <= 1:
        return [fn(*a) for a in args]
    with cf.ProcessPoolExecutor(workers, mp_context=multiprocessing.get_context("spawn")) as ex:
        return list(ex.map(fn, *zip(*args), chunksize=max(1, len(args) // (4 * workers))))


def _scaled(rng, n, rho):
    A = rng.normal(size=(n, n))
    return A * (rho / np.max(np.abs(np.linalg.eigvals(A))))


def gram_plants():
    """(name, A, B, Q, R, horizons): the plants of the Gram-extreme checks. Spectral radii 0.5 .. 1.5 with the sweep's
    own plant; m = 1, 2, 4; a nearly uncontrollable B (one column 1e-6), B columns 1e4 apart, a strongly non-normal A;
    non-scalar Q, R (time-major convention) with cond up to 1e6. Large N m is kept to a few cases (the 50-digit
    eigen-solve of an N m = 100 matrix takes seconds)."""
    rng = np.random.default_rng(20261020)
    out = [("sweep", SWEEP_A, SWEEP_B, SWEEP_Q, SWEEP_R, GRAM_HORIZONS)]
    for rho in (0.5, 0.999, 1.117, 1.3, 1.5):
        out.append(("n2m1_rho%g" % rho, _scaled(rng, 2, rho), rng.normal(size=(2, 1)), 2.0 * np.eye(2), np.eye(1),
                    GRAM_HORIZONS))
        out.append(("n2m2_rho%g" % rho, _scaled(rng, 2, rho), rng.normal(size=(2, 2)), 1.5 * np.eye(2),
                    0.7 * np.eye(2), (1, 2, 12, 13, 30) + ((50,) if rho in (1.117, 1.5) else ())))
    out.append(("n4m4_rho1.3", _scaled(rng, 4, 1.3), rng.normal(size=(4, 4)), np.eye(4), np.eye(4), (1, 2, 12, 13)))
    out.append(("n3m1_rho1.25", _scaled(rng, 3, 1.25), rng.normal(size=(3, 1)), np.eye(3), np.eye(1), (13, 40)))
    B = rng.normal(size=(2, 2)); B[:, 1] *= 1e-6
    out.append(("uncontrollable_col", _scaled(rng, 2, 1.117), B, 2.0 * np.eye(2), np.eye(2), (1, 12, 30)))
    B = rng.normal(size=(2, 2)); B[:, 0] *= 1e2; B[:, 1] *= 1e-2
    out.append(("cols_1e4_apart", _scaled(rng, 2, 1.117), B, 2.0 * np.eye(2), np.eye(2), (2, 13, 30)))
    out.append(("non_normal", np.array([[0.9, 40.0], [0.0, 0.95]]), np.array([[0.0], [1.0]]), np.eye(2), np.eye(1),
                (2, 12, 30, 50)))
    Uq, _ = np.linalg.qr(rng.normal(size=(2, 2)))
    Qg = Uq @ np.diag([1e3, 1e-3]) @ Uq.T                  # cond(Q) = 1e6
    Ur, _ = np.linalg.qr(rng.normal(size=(2, 2)))
    Rg = Ur @ np.diag([10.0, 0.1]) @ Ur.T                  # cond(R) = 1e2
    out.append(("weights_cond1e6", _scaled(rng, 2, 1.3), rng.normal(size=(2, 2)), Qg, Rg, (1, 13, 30)))
    Uq3, _ = np.linalg.qr(rng.normal(size=(3, 3)))
    out.append(("weights_n3m2", _scaled(rng, 3, 1.117), rng.normal(size=(3, 2)), Uq3 @ np.diag([1e2, 1.0, 1e-4])
                @ Uq3.T, np.array([[2.0, 0.9], [0.9, 1.0]]), (2, 12, 30)))
    return out


def gram_perturbations(name, n, m, S=2):
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    return 1e-3 * rng.uniform(-1, 1, size=(n * n, S)), 1e-3 * rng.uniform(-1, 1, size=(n * m, S))


def model(A, B, dA, dB, s):
    n, m = B.shape
    return A + dA[:, s].reshape(n, n), B + dB[:, s].reshape(n, m)


def gram_truth_float(Ah, Bh, Q, R, N, strict):
    g = mt.gram_truth(Ah, Bh, Q, R, N, strict)
    return {k: float(v) for k, v in g.items()}


def assert_gram(min_H, norm_Gamma, truth, tol=GRAM_TOL, what=""):
    """Relative errors of min_H and norm_Gamma^2 against the truth; returns (err_min_H, err_cmax)."""
    e_h = abs(min_H - truth["min_H"]) / abs(truth["min_H"])
    e_c = abs(norm_Gamma ** 2 - truth["cmax"]) / truth["cmax"]
    assert e_h <= tol and e_c <= tol, (what, e_h, e_c, tol)
    return e_h, e_c


def dense_tol(N, m, cond_H):
    """Tolerance of the dense route (Gram matrix assembled in float64, Householder tridiagonalisation, Sturm bisection):
    the computed tridiagonal is exactly similar to H^ + E with ||E||_2 <= c u ||H^||_2 (Wilkinson's backward-error bound
    for k - 2 Householder reflections of a k x k matrix, k = N m, plus the rounding of the assembled entries, each a sum
    of at most (N + 1) n products), so by Weyl lambda_min moves by at most c u lambda_max(H^), i.e. by c u cond(H^)
    relative. c = 4 k covers the reflector count with the factor of a few that the analysis carries per reflector."""
    return max(1e-9, 4.0 * N * m * U * cond_H)


# ------------------------------------------------------------------------------------------------ whole chain
def truth_sample(Ah, Bh, Q, R, lo, hi, N, e, MV, x, V_expert, strict=True, K=None, gram=True):
    """k3_truth of one sample reduced to floats: fields, kappa, expected flags, ceil distances."""
    t = mt.k3_truth(Ah, Bh, Q, R, lo, hi, N, e, e, MV, x, P3, V_expert, strict, K=K,
                    gram=None if gram else False, kappa=gram)
    b32, b512 = mt.k3_expected_flags(t, EDGE_MARGIN)
    f = {k: float(v) for k, v in t["fields"].items()}
    return {"fields": f, "kappa": {k: float(v) for k, v in t["kappa"].items()}, "b32": b32, "b512": b512,
            "raises": t["raises"], "den": float(t["edges"]["den"]),
            "ceil_dist": {k: float(v) for k, v in t["ceil_dist"].items()},
            "ceil_margin": {"N_0": 1e-9 * (1 + abs(float(t["edges"]["N0_arg"])) if mp.isfinite(t["edges"]["N0_arg"])
                                          else 1.0) * (1 + abs(f["gamma"]) if np.isfinite(f["gamma"]) else 1.0),
                            "N_min": 1e-9 * (1 + abs(float(t["edges"]["Nmin_arg"])) if mp.isfinite(
                                t["edges"]["Nmin_arg"]) else 1.0) * (1 + abs(f["gamma"]) if np.isfinite(f["gamma"])
                                                                     else 1.0)},
            "cond_H": float(t["cond_H"])}


INTEGER_FIELDS = ("N_0", "N_min")
GRAM_FIELDS = ("min_H", "norm_Gamma")


def compare_fields(got, t, gram_tol=GRAM_TOL, fields=mt.BOUND_FIELDS):
    """got: field -> float of one sample. Every field the truth defines must be within FIELD_TOL (1 + kappa) (the Gram
    extremes within gram_tol); N_0 / N_min equal unless the truth is within rounding of a ceil jump. Returns
    (max relative error per field, number of ceil-edge samples skipped)."""
    errs, skipped = {}, 0
    f = t["fields"]
    for k in fields:
        v = f[k]
        if k in INTEGER_FIELDS:
            if not np.isfinite(v):
                continue
            if got[k] != v:
                assert t["ceil_dist"][k] <= t["ceil_margin"][k], (k, got[k], v, t["ceil_dist"][k])
                skipped += 1
            continue
        if not np.isfinite(v):
            continue
        assert np.isfinite(got[k]), (k, got[k], v)
        err = abs(got[k] - v) / max(abs(v), 1e-300)
        tol = gram_tol if k in GRAM_FIELDS else FIELD_TOL * (1.0 + t["kappa"][k])
        assert err <= tol, (k, got[k], v, err, tol)
        errs[k] = err / (1.0 + t["kappa"][k]) if k not in GRAM_FIELDS else err
    return errs, skipped


def check_flags(flags, truths):
    """Bits 32 and 512 against the truth in both directions; returns the number of edge samples (either value
    allowed)."""
    edge = 0
    for fl, t in zip(flags, truths):
        fl = int(fl)
        for bit, want in ((32, t["b32"]), (512, t["b512"])):
            if want is None:
                edge += 1
            else:
                assert bool(fl & bit) == want, (bit, fl, want, t["den"], t["raises"])
    return edge


def pick_decisive(fields_by_name, rng, n_edge, n_random):
    """Indices of a batch chosen on purpose from the float64 results of the whole batch: the smallest
    |1 - xi - eta| / (1 + |xi| + |eta|), the smallest |sqrt(err_th) argument| relative, the nearest to N_0's ceil
    jump, plus random ones."""
    g = fields_by_name
    S = len(g["xi"])
    xi, eta, w05, w1 = g["xi"], g["eta"], g["omega_N0d5"], g["omega_N1"]
    with np.errstate(all="ignore"):
        den = np.abs(1 - xi - eta) / (1 + np.abs(xi) + np.abs(eta))
        disc = np.abs(w05 ** 2 + w1 * (1 - eta)) / (w05 ** 2 + np.abs(w1 * (1 - eta)))
        n0 = g["L_V"] - g["gamma"]                 # M_V / eps - gamma where that is the larger one
        frac = np.where(n0 > 0, np.abs(n0 - np.round(n0)), np.inf)
    picks = []
    for key in (den, disc, frac):
        key = np.where(np.isfinite(key), key, np.inf)
        picks.extend(int(i) for i in np.argsort(key, kind="stable")[:n_edge])
    picks.extend(int(i) for i in rng.choice(S, size=min(n_random, S), replace=False))
    return sorted(set(picks))


def place_gain(A, B, poles):
    """u = +K x placing the closed-loop poles of a single-input pair (Ackermann)."""
    n = A.shape[0]
    C = np.hstack([np.linalg.matrix_power(A, k) @ B for k in range(n)])
    coef = np.poly(poles)
    phi = sum(c * np.linalg.matrix_power(A, n - i) for i, c in enumerate(coef))
    e = np.zeros(n); e[-1] = 1.0
    return -(e @ np.linalg.solve(C, phi)).reshape(1, n)


def edge_cases():
    """Samples of the sweep plant straddling each classification edge: (tag, dA, dB, N, e, M_V, K or None).
      den     1 - xi - eta = 0, by scaling e around the root e* = sqrt(err_th / (1 / minQ + 1 / minR)) of xi(e) = 1 - eta;
      rho_cl  rho(A^ + B^K) = 0.6 (rho_K = 1, gamma changes sign), by an explicit gain placing the poles at 0.6 (1 +- d);
      arg1    A^ = 0: the argument of math.log is exactly 0;
      sqrt    gamma < 0 with M_V below / above epsilon_K (omega_N0d5's first sqrt argument changes sign) and small N
              with eta > 1 (err_th's argument negative)."""
    n, m = 2, 1
    z4, z2 = np.zeros(4), np.zeros(2)
    out = []
    rel = (1e-2, 1e-4, 1e-7, 1e-10, 1e-13)
    for N in (7, 12):
        t = mt.k3_truth(SWEEP_A, SWEEP_B, SWEEP_Q, SWEEP_R, SWEEP_LO, SWEEP_HI, N, 5e-3, 5e-3, 0.05, [0.15, 0.1],
                        P3, 0.3, True, gram=False, kappa=False)
        e_star = float(mp.sqrt(t["fields"]["err_th"] / (1 / mp.mpf(2) + 1)))
        for d in rel:
            for sgn in (-1, 1):
                out.append(("den", z4, z2, N, e_star * (1 + sgn * d), 0.05, None))
    for d in (1e-2, 1e-5, 1e-9, 1e-13):
        for sgn in (-1, 1):
            K = place_gain(SWEEP_A, SWEEP_B, [0.6 * (1 + sgn * d), 0.3])
            for N in (3, 20):
                out.append(("rho_cl", z4, z2, N, 5e-3, 0.05, K))
    out.append(("arg1", -SWEEP_A.reshape(-1), z2, 5, 5e-3, 0.05, None))
    Kun = place_gain(SWEEP_A, SWEEP_B, [0.7, 0.3])            # rho_cl = 0.7: gamma < 0
    for MV in (1e-6, 1e-2, 10.0):
        out.append(("sqrt", z4, z2, 6, 5e-3, MV, Kun))
    for N in (1, 2, 3, 4):
        for MV in (0.01, 0.5, 3.0):
            out.append(("sqrt", z4, z2, N, 5e-3, MV, None))
    return out
