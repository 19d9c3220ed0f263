"""CPU tier — the horizon-range numerics of K2a and K3 (clqr.cuh: plan_prepare_range + the stage-offset solve;
bounds.cuh / gramspec.cuh: bounds_prefix + gram_spectrum_range) against their single-horizon counterparts, compiled
with g++ from the engine headers into a test-only library (tests/hostmath/range.cpp, the flags of
tests/hostmath/build.py). The GPU tier (tests/test_horizon_range.py) repeats the comparisons through the C ABI.
"""
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import pytest

from oracle import np_sampler

HERE = os.path.dirname(os.path.abspath(__file__))
HM = os.path.join(HERE, "hostmath")
CSRC = os.path.join(os.path.dirname(HERE), "lq_mpc_b200", "csrc")
COMPILED_DIMS = [(1, 1), (2, 1), (2, 2), (3, 1), (3, 2), (3, 3), (4, 1), (4, 2), (4, 4), (6, 2), (8, 2)]
BOUND_FIELDS = ['alpha', 'beta', 'xi', 'eta', 'bound', 'E_psi', 'E_u', 'E_psi_u', 'theta_u', 'theta_x_u', 'C_K',
                'rho_K', 'gamma', 'rho_gamma', 'L_V', 'N_0', 'omega_N1', 'omega_N0d5', 'err_th', 'N_min', 'h',
                'epsilon_K', 'norm_A', 'norm_B', 'norm_K', 'norm_Gamma', 'norm_Phi', 'min_H', 'rho_cl', 'bar_u',
                'bar_d_u']
# fields that depend on the two Gram-spectrum extremes (bisection results: agree to the search tolerance); every other
# field, the error-consistent sums included, is computed by the same operations in both forms and must be bit-equal
GRAM_FIELDS = {'alpha', 'beta', 'bound', 'E_u', 'E_psi_u', 'theta_u', 'theta_x_u', 'norm_Gamma', 'min_H'}
HORIZON_FREE = ['epsilon_K', 'norm_A', 'norm_B', 'norm_K', 'rho_cl', 'bar_u', 'bar_d_u', 'C_K', 'rho_K', 'gamma',
                'rho_gamma', 'h']
TOL = 1e-9

_P = ctypes.POINTER(ctypes.c_double)
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(HM, "_build")
        os.makedirs(out, exist_ok=True)
        so = os.path.join(out, "librange.so")
        src = os.path.join(HM, "range.cpp")
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


def mpc(rng_mode, A, B, Q, R, lo, hi, dA, dB, Nmin, Nmax, pts=None, x0=None):
    """rng_mode 1: range form, 0: one single-horizon solve per N. Returns V [H][P][S], u0, M_V [H][S], flags."""
    n, m = B.shape
    S = dA.shape[1]
    H = Nmax - Nmin + 1
    P = pts.shape[0] if pts is not None else 1
    keep = [_c(a) for a in (A, B, Q, R, Q, lo, hi, dA, dB, pts, x0)]
    o = {"V": np.zeros((H, P, S)), "u0": np.zeros((H, P, m, S)), "M_V": np.zeros((H, S)),
         "flags": np.zeros((H, P, S), dtype=np.int32)}
    rc = lib().hr_mpc(rng_mode, n, m, *[_p(a) for a in keep[:7]], ctypes.c_int64(S), _p(keep[7]), _p(keep[8]), Nmin,
                      Nmax, P, _p(keep[9]), _p(keep[10]), _p(o["V"]), _p(o["u0"]), _p(o["M_V"]),
                      o["flags"].ctypes.data_as(ctypes.POINTER(ctypes.c_int32)))
    assert rc == 0
    return o


def bounds(rng_mode, A, B, Q, R, lo, hi, dA, dB, Nmin, Nmax, e, MV, x, p, Vexp):
    n, m = B.shape
    S = dA.shape[1]
    H = Nmax - Nmin + 1
    keep = [_c(a) for a in (A, B, Q, R, Q, lo, hi, dA, dB, e, e, MV, x, p)]
    detail = np.zeros((H, len(BOUND_FIELDS), S))
    flags = np.zeros((H, S), dtype=np.int32)
    stages = np.zeros(S, dtype=np.int64)
    probes = np.zeros((H, S), dtype=np.int32)
    rc = lib().hr_bounds(rng_mode, n, m, *[_p(a) for a in keep[:7]], ctypes.c_int64(S), _p(keep[7]), _p(keep[8]),
                         Nmin, Nmax, *[_p(a) for a in keep[9:]], ctypes.c_double(Vexp), _p(detail),
                         flags.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
                         stages.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)),
                         probes.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)))
    assert rc == 0
    return {"detail": detail, "flags": flags, "stages": stages, "probes": probes}


def bits(a):
    return np.ascontiguousarray(a).view(np.int64 if a.dtype == np.float64 else a.dtype)


def assert_mpc_bit_equal(r, s):
    for k in ("V", "u0", "M_V", "flags"):
        assert np.array_equal(bits(r[k]), bits(s[k])), k


def assert_bounds_agree(r, s):
    assert np.array_equal(r["flags"], s["flags"])
    for i, f in enumerate(BOUND_FIELDS):
        a, b = r["detail"][:, i], s["detail"][:, i]
        if f in GRAM_FIELDS:
            fin = np.isfinite(b)
            assert np.array_equal(np.isfinite(a), fin), f
            err = np.abs(a[fin] - b[fin]) / np.maximum(np.abs(b[fin]), 1e-300)
            assert err.size == 0 or err.max() <= TOL, (f, err.max())
        else:
            assert np.array_equal(bits(a), bits(b)), f
    for f in HORIZON_FREE:                      # one value per sample, whatever the horizon
        col = r["detail"][:, BOUND_FIELDS.index(f)]
        assert np.array_equal(bits(col), bits(np.broadcast_to(col[:1], col.shape))), f


def level4_perturbations(count, error_vec):
    """The first `count` perturbations of level index 4 of cfg-sweep-f's seeded grids (seed 20240522)."""
    n_boundary = count // 5
    gA, _, _ = np_sampler.sample_error_grid(20240522, 0, 2, 2, count, error_vec, n_boundary, "f")
    gB, _, _ = np_sampler.sample_error_grid(20240522, 1, 2, 1, count, error_vec, n_boundary, "f")
    return (np.ascontiguousarray(gA[:, :, :, 4]).reshape(4, count),
            np.ascontiguousarray(gB[:, :, :, 4]).reshape(2, count))


@pytest.fixture(scope="module")
def golden_setup(example, known):
    A, B, Q, R, lo, hi = (example[x] for x in ("A", "B", "Q", "R", "lo", "hi"))
    ring = np.array(known["single"]["x0_vec"])
    return A, B, Q, R, lo, hi, ring


def test_range_ring_solves_bit_identical_golden(golden_setup, golden):
    A, B, Q, R, lo, hi, ring = golden_setup
    eA = np.ascontiguousarray(golden["error_A_f"][:, :, :40, 4]).reshape(4, -1)
    eB = np.ascontiguousarray(golden["error_B_f"][:, :, :40, 4]).reshape(2, -1)
    assert_mpc_bit_equal(mpc(1, A, B, Q, R, lo, hi, eA, eB, 1, 50, pts=ring.T),
                         mpc(0, A, B, Q, R, lo, hi, eA, eB, 1, 50, pts=ring.T))
    x0 = np.random.default_rng(7).uniform(-3, 3, size=(2, eA.shape[1]))
    assert_mpc_bit_equal(mpc(1, A, B, Q, R, lo, hi, eA, eB, 3, 50, x0=x0),
                         mpc(0, A, B, Q, R, lo, hi, eA, eB, 3, 50, x0=x0))


def test_range_bounds_golden_and_fewer_stages(golden_setup, known, example):
    """N = 1..50 on the first 1 000 level-4 perturbations of cfg-sweep-f: every field within 1e-9 of the
    single-horizon computation (the horizon-independent ones bit-equal), equal flags, and the range search runs
    fewer elimination stages than the 50 per-horizon searches."""
    A, B, Q, R, lo, hi, ring = golden_setup
    error_vec = np.linspace(1e-3, 1e-2, 10)
    eA, eB = level4_perturbations(1000, error_vec)
    S = eA.shape[1]
    x_start = ring[:, 1]
    mv = mpc(1, A, B, Q, R, lo, hi, eA, eB, 1, 50, pts=ring.T)["M_V"]
    e = np.full(S, error_vec[4])
    xs = np.repeat(x_start[:, None], S, axis=1)
    V_exp = 0.3
    r = bounds(1, A, B, Q, R, lo, hi, eA, eB, 1, 50, e, mv, xs, example["p"], V_exp)
    s = bounds(0, A, B, Q, R, lo, hi, eA, eB, 1, 50, e, mv, xs, example["p"], V_exp)
    assert_bounds_agree(r, s)
    # per-horizon searches: the range search with N_min == N_max is gram_spectrum itself (its extremes are bit-equal
    # to those of bounds_sample), so its stage count is that of the single-horizon search
    per_stages = np.zeros(S, dtype=np.int64)
    gram = [BOUND_FIELDS.index("min_H"), BOUND_FIELDS.index("norm_Gamma")]
    for N in range(1, 51):
        one = bounds(1, A, B, Q, R, lo, hi, eA, eB, N, N, e, mv[N - 1:N], xs, example["p"], V_exp)
        assert np.array_equal(bits(one["detail"][0][gram]), bits(s["detail"][N - 1][gram]))
        per_stages += one["stages"]
    ratio = per_stages.sum() / r["stages"].sum()
    print("elimination stages: per-horizon %d, range %d, ratio %.2f" % (per_stages.sum(), r["stages"].sum(), ratio))
    assert ratio > 1.0


@pytest.mark.parametrize("n,m", COMPILED_DIMS)
def test_range_every_compiled_pair(n, m):
    """Random stabilisable models with a saturating box: range ring solves bit-equal to the single-horizon ones (ring
    points and per-sample states, N_min > 1, N_min == N_max), bounds within 1e-9 with equal flags."""
    rng = np.random.default_rng(100 * n + m)
    A = rng.normal(size=(n, n))
    A *= 1.05 / max(np.max(np.abs(np.linalg.eigvals(A))), 1e-3)
    B = rng.normal(size=(n, m))
    M = rng.normal(size=(n, n)); Q = M @ M.T + 0.5 * np.eye(n)
    M = rng.normal(size=(m, m)); R = M @ M.T + 0.5 * np.eye(m)
    lo, hi = -0.3 * np.ones(m), 0.4 * np.ones(m)
    S = 6
    dA = 0.01 * rng.normal(size=(n * n, S))
    dB = 0.01 * rng.normal(size=(n * m, S))
    pts = rng.uniform(-2, 2, size=(3, n))
    x0 = rng.uniform(-2, 2, size=(n, S))
    Nmax = 18 if n <= 4 else 10
    for Nmin, Nx in ((3, Nmax), (Nmax, Nmax)):
        assert_mpc_bit_equal(mpc(1, A, B, Q, R, lo, hi, dA, dB, Nmin, Nx, pts=pts),
                             mpc(0, A, B, Q, R, lo, hi, dA, dB, Nmin, Nx, pts=pts))
        assert_mpc_bit_equal(mpc(1, A, B, Q, R, lo, hi, dA, dB, Nmin, Nx, x0=x0),
                             mpc(0, A, B, Q, R, lo, hi, dA, dB, Nmin, Nx, x0=x0))
    # scalar weights: the matrix-free route the range kernel takes (also with non-scalar ones, strict_reference = 0)
    Qs, Rs = 2.0 * np.eye(n), np.eye(m)
    H = Nmax - 1
    mv = rng.uniform(1.0, 5.0, size=(H, S))
    e = np.full(S, 5e-3)
    r = bounds(1, A, B, Qs, Rs, lo, hi, dA, dB, 2, Nmax, e, mv, x0, np.array([0.1, 1, 0.6]), 0.3)
    s = bounds(0, A, B, Qs, Rs, lo, hi, dA, dB, 2, Nmax, e, mv, x0, np.array([0.1, 1, 0.6]), 0.3)
    assert_bounds_agree(r, s)


@pytest.mark.parametrize("e", [1e-7, 1e-8])
def test_range_bounds_tiny_error_levels(golden_setup, example, e):
    """Error levels far below the sweep's: (e_A + ||A^||)^i - ||A^||^i cancels almost completely, so the error-consistent
    sums of the range form must be built from the same terms as the single-horizon ones, not from running products."""
    A, B, Q, R, lo, hi, ring = golden_setup
    rng = np.random.default_rng(11)
    S = 200
    eA = e * rng.uniform(-1, 1, size=(4, S))
    eB = e * rng.uniform(-1, 1, size=(2, S))
    mv = mpc(1, A, B, Q, R, lo, hi, eA, eB, 1, 50, pts=ring.T)["M_V"]
    ev = np.full(S, e)
    xs = np.repeat(ring[:, 1:2], S, axis=1)
    r = bounds(1, A, B, Q, R, lo, hi, eA, eB, 1, 50, ev, mv, xs, example["p"], 0.3)
    s = bounds(0, A, B, Q, R, lo, hi, eA, eB, 1, 50, ev, mv, xs, example["p"], 0.3)
    assert_bounds_agree(r, s)
