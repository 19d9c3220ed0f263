"""CPU tier — the ENGINE'S OWN per-sample math (the __host__ __device__ templates under lq_mpc_b200/csrc/*.cuh that
the sm_100a kernels instantiate) compiled with g++ into a TEST-ONLY harness (tests/hostmath) and compared with the
oracle and the golden vectors in the GPU-less build container. This is not a CPU path of the product: nothing under
lq_mpc_b200/ loads the harness, and the harness has no SoA pipeline, no reductions and no ABI.
The GPU tier (tests/test_gpu_parity.py) repeats the comparisons through the C ABI on the real kernels.
"""
import numpy as np
import pytest

from oracle import np_batched as nb
from oracle import np_oracle as o
from tests.conftest import relerr

hm = pytest.importorskip("tests.hostmath.api")
TOL = 1e-9
# every (n, m) the engine instantiates its templates for (LQ_FOR_EACH_DIM in lq_mpc_b200/csrc/engine.h)
COMPILED_DIMS = [(1, 1), (2, 1), (2, 2), (3, 1), (3, 2), (3, 3), (4, 1), (4, 2), (4, 4), (6, 2), (8, 2)]


@pytest.mark.parametrize("n", [1, 2, 3, 4, 6, 8])
def test_spectral_radius_vs_lapack(n):
    rng = np.random.default_rng(n)
    M = rng.normal(size=(300, n, n))
    M[:20] *= 1e-3
    M[20:40] *= 1e3
    if n >= 2:
        M[40] = np.eye(n)                                  # repeated eigenvalue
        M[41] = np.triu(np.ones((n, n)))                   # defective (Jordan-like)
        M[42] = 0.0
        M[43] = np.diag(np.arange(1, n + 1.0))
        rot = np.eye(n); rot[:2, :2] = [[0, -1], [1, 0]]   # eigenvalues on the unit circle
        M[44] = rot
    rho, ok = hm.spectral_radius(M)
    ref = np.max(np.abs(np.linalg.eigvals(M)), axis=1)
    assert np.all(ok == 1)
    scale = np.maximum(ref, 1e-12 * np.linalg.norm(M, axis=(1, 2)))
    err = np.abs(rho - ref) / np.where(scale > 0, scale, 1.0)
    err[41] = min(err[41], 1e-12) if abs(rho[41] - 1.0) < 1e-4 else err[41]   # defective: sqrt(eps)-conditioned
    assert err.max() < 1e-10, (int(err.argmax()), err.max())


@pytest.mark.parametrize("n", [3, 4])
def test_closed_form_spectral_radius_is_trusted_only_when_accurate(n):
    """eig.cuh fast path (characteristic polynomial -> Ferrari -> Bairstow polish -> conditioning test) alone:
    whatever it ACCEPTS must be within 1e-10 of LAPACK (the QR iteration takes the rest); generic matrices are
    accepted, clustered spectra are not."""
    rng = np.random.default_rng(10 + n)
    S = 60_000
    fam = {"gauss": rng.normal(size=(S, n, n)),
           "scaled": rng.normal(size=(S, n, n)) * np.exp(rng.uniform(-3, 3, size=(S, n, 1))),
           "sym": (lambda M: M + M.transpose(0, 2, 1))(rng.normal(size=(S, n, n))),
           "cluster": 0.9 * np.eye(n)[None] + 0.02 * rng.normal(size=(S, n, n)),
           "tight": 0.9 * np.eye(n)[None] + 1e-3 * rng.normal(size=(S, n, n)),
           "huge_range": rng.normal(size=(S, n, n)) * 10.0 ** rng.integers(-100, 100, size=(S, 1, 1))}
    for name, M in fam.items():
        rho, ok = hm.spectral_radius_poly(M)
        ref = np.max(np.abs(np.linalg.eigvals(M)), axis=1)
        tr = ok == 1
        if tr.any():
            assert np.max(np.abs(rho[tr] - ref[tr]) / ref[tr]) < 1e-10, name
        if name in ("gauss", "sym", "huge_range"):
            assert tr.mean() > 0.999, (name, tr.mean())
        if name == "tight":
            assert tr.mean() < 0.01, (name, tr.mean())
        full, okf = hm.spectral_radius(M)                      # dispatcher = fast path or QR fallback
        assert np.all(okf == 1) and np.max(np.abs(full - ref) / ref) < 1e-9, name
    z, okz = hm.spectral_radius_poly(np.zeros((3, n, n)))
    assert np.all(z == 0.0) and np.all(okz == 1)


@pytest.mark.parametrize("n,m,e", [(4, 2, 0.01), (2, 1, 0.05), (1, 1, 0.1), (3, 2, 0.3), (3, 3, 0.1), (4, 1, 0.05),
                                   (4, 4, 0.2), (6, 2, 0.05), (8, 2, 0.02), (2, 2, 0.1), (3, 1, 0.1)])
def test_k1_math_vs_batched_oracle(n, m, e):
    A, B, Q, R = nb.synth_problem(n, m, seed=0)
    S = 257
    dA, dB, x0 = nb.synth_samples(n, m, S, seed=1, e=e)
    Pexp = nb.expert_matrix(A, B, Q, R, Q, 30)
    ref = nb.eval_batch(A, B, Q, R, Q, Pexp, dA, dB, x0, 2, 11, T=25, want_K=True)
    got = hm.eval_batch(A, B, Q, R, Q, 30, *nb.to_soa(dA, dB, x0), 2, 11, 25)
    assert relerr(got["prep"][:n * n].reshape(n, n), Pexp) < 1e-12
    well = np.abs(ref["rho"] - 1.0) > 1e-6
    assert np.array_equal((got["flags"] & 1) != 0, ref["unstable"])
    for k, kr in (("rho", "rho"), ("V_N", "Vn"), ("J_T", "JT")):
        assert relerr(got[k], ref[kr]) < TOL, k
    for k in ("J", "ratio"):
        assert relerr(np.where(well, got[k], 0.0), np.where(well, ref[k], 0.0)) < 1e-8, k
    K = got["K0"].reshape(10, m, n, S).transpose(0, 3, 1, 2)
    assert np.max(np.abs(K - ref["K0"])) < 1e-10 * max(1.0, np.max(np.abs(ref["K0"])))
    assert not np.any(got["flags"] & ~1)


def test_k2_math_mpc_test_and_random_api(known):
    """Exact box-constrained solves / closed loops vs the untouched reference's answers."""
    k = known["mpc_test"]
    A = np.array([[1, 0.7], [0.12, 0.4]]); B = np.array([[1], [1.2]])
    Q = 2 * np.eye(2); R = np.eye(1); lo, hi = np.array([-0.1]), np.array([0.1])
    x0 = np.array([[0.1125], [0.19]])
    sol = hm.mpc(0, A, B, Q, R, Q, lo, hi, None, None, 20, x0_soa=x0)
    assert abs(sol["V"][0, 0] - k["V_N"]) < TOL * k["V_N"] and abs(sol["u0"][0, 0, 0] - k["u_0"][0]) < 1e-12
    assert sol["flags"][0, 0] == 2
    dA = (np.array([[1.01, 0.7], [0.12, 0.41]]) - A).reshape(4, 1)
    dB = (np.array([[1], [1.21]]) - B).reshape(2, 1)
    # plant = (A_true, B_true) is the PROBLEM; the controller model is plant + (A - A_true)
    At, Bt = A + dA.reshape(2, 2), B + dB.reshape(2, 1)
    sim = hm.mpc(1, At, Bt, Q, R, Q, lo, hi, -dA, -dB, 6, T=20, x0_soa=x0)
    assert abs(sim["J_T"][0] - k["J_T"]) < TOL * k["J_T"]
    assert np.max(np.abs(sim["X"][:, :, 0].T - np.array(k["X"]))) < 1e-12
    assert np.max(np.abs(sim["U"][:, :, 0].T - np.array(k["U"]))) < 1e-12
    for c in known["random_api"]:
        n, m, N, T = c["n"], c["m"], c["N"], c["T"]
        A, B, dA, dB = (np.array(c[x]) for x in ("A", "B", "dA", "dB"))
        Q, R = c["q"] * np.eye(n), c["r"] * np.eye(m)
        lo, hi = -c["ub"] * np.ones(m), c["ub"] * np.ones(m)
        x0 = np.array(c["x0"]).reshape(n, 1)
        sol = hm.mpc(0, A, B, Q, R, Q, lo, hi, dA.reshape(-1, 1), dB.reshape(-1, 1), N, x0_soa=x0)
        assert abs(sol["V"][0, 0] - c["V_N"]) < TOL * abs(c["V_N"])
        assert np.max(np.abs(sol["u0"][0, :, 0] - np.array(c["u_0"]))) < 1e-10
        sim = hm.mpc(1, A, B, Q, R, Q, lo, hi, dA.reshape(-1, 1), dB.reshape(-1, 1), N, T=T, x0_soa=x0)
        assert abs(sim["J_T"][0] - c["J_T"]) < TOL * abs(c["J_T"])
        assert np.max(np.abs(sim["U"][:, :, 0].T - np.array(c["U"]))) < 1e-10


def test_k2_math_tracking_references(tracking):
    """The affine (non-zero reference) branch of the exact solver vs the untouched reference's answers, then a batch
    of random references vs the oracle's dense QP (saturated and unsaturated mixed)."""
    from tests.conftest import tracking_case
    for c in map(tracking_case, tracking):
        n = c["n"]
        a = (c["A"], c["B"], c["Q"], c["R"], c["Q"], c["lo"], c["hi"], c["dA"].reshape(-1, 1), c["dB"].reshape(-1, 1))
        sol = hm.mpc(0, *a, c["N"], x0_soa=c["x0"].reshape(n, 1), x_ref=c["x_ref"], u_ref=c["u_ref"])
        assert abs(sol["V"][0, 0] - c["V_N"]) < TOL * abs(c["V_N"])
        assert np.max(np.abs(sol["u0"][0, :, 0] - c["u_0"])) < 1e-10
        sim = hm.mpc(1, *a, c["N"], T=c["T"], x0_soa=c["x0"].reshape(n, 1), x_ref=c["x_ref"], u_ref=c["u_ref"])
        assert abs(sim["J_T"][0] - c["J_T"]) < TOL * abs(c["J_T"])
        assert np.max(np.abs(sim["U"][:, :, 0].T - c["U"])) < 1e-10
        assert np.max(np.abs(sim["X"][:, :, 0].T - c["X"])) < 1e-10
    rng = np.random.default_rng(5)
    n, m, N, S = 4, 2, 6, 64
    A = rng.normal(size=(n, n)); A *= 0.9 / np.max(np.abs(np.linalg.eigvals(A)))
    B = rng.normal(size=(n, m)); Q = np.eye(n); R = 0.5 * np.eye(m)
    lo, hi = -0.3 * np.ones(m), 0.3 * np.ones(m)
    dA = rng.uniform(-0.01, 0.01, size=(n * n, S)); dB = rng.uniform(-0.01, 0.01, size=(n * m, S))
    x0 = rng.normal(size=(n, S)) * 0.5
    for xr, ur in ((rng.normal(size=(n, N)) * 0.3, None), (None, rng.normal(size=(m, N)) * 0.2),
                   (rng.normal(size=(n, N + 3)) * 0.3, rng.normal(size=(m, N + 3)) * 0.2)):
        sol = hm.mpc(0, A, B, Q, R, Q, lo, hi, dA, dB, N, x0_soa=x0, x_ref=xr, u_ref=ur)
        n_act = 0
        for s in range(S):
            u0, V, act = o.mpc_solve(N, A + dA[:, s].reshape(n, n), B + dB[:, s].reshape(n, m), Q, R, Q, lo, hi,
                                     x0[:, s], x_ref=xr, u_ref=ur)
            n_act += int(act)
            assert abs(sol["V"][0, s] - V) < TOL * abs(V) and np.max(np.abs(sol["u0"][0, :, s] - u0)) < 1e-9
            assert bool(sol["flags"][0, s] & 2) == act
        assert 0 < n_act < S


def test_k2_math_general_polytope(polytope):
    """pclqr.cuh (stage-wise projected Riccati sweeps) vs the untouched reference's answers, vs the dense active-set
    oracle on random polytopes (m = 1..4, up to 9 rows), bit-level agreement with the box solver when the polytope IS
    a box, and a degenerate polytope (duplicate + redundant rows, three rows through one vertex) with references."""
    from tests.conftest import polytope_case, random_polytope
    for c in map(polytope_case, polytope):
        n = c["n"]
        a = (c["A"], c["B"], c["Q"], c["R"], c["Q"], None, None, c["dA"].reshape(-1, 1), c["dB"].reshape(-1, 1))
        sol = hm.mpc(0, *a, c["N"], x0_soa=c["x0"].reshape(n, 1), F_u=c["F_u"])
        assert abs(sol["V"][0, 0] - c["V_N"]) < TOL * abs(c["V_N"])
        assert np.max(np.abs(sol["u0"][0, :, 0] - c["u_0"])) < 1e-10
        sim = hm.mpc(1, *a, c["N"], T=c["T"], x0_soa=c["x0"].reshape(n, 1), F_u=c["F_u"])
        assert abs(sim["J_T"][0] - c["J_T"]) < TOL * abs(c["J_T"])
        assert np.max(np.abs(sim["U"][:, :, 0].T - c["U"])) < 1e-10 and not (sim["flags"][0, 0] & ~2)
    rng = np.random.default_rng(7)
    n_act = tot = 0
    for n, m, p in [(2, 1, 2), (2, 2, 3), (2, 2, 5), (3, 2, 6), (4, 2, 8), (3, 3, 6), (4, 4, 8), (3, 3, 9)]:
        for rep in range(2):
            N = int(rng.integers(2, min(12, 128 // p) + 1))
            A = rng.normal(size=(n, n)); A *= rng.uniform(0.6, 1.2) / np.max(np.abs(np.linalg.eigvals(A)))
            B = rng.normal(size=(n, m)); Q = rng.uniform(0.5, 3) * np.eye(n); R = rng.uniform(0.1, 2) * np.eye(m)
            if rep:
                Mq, Mr = rng.normal(size=(n, n)), rng.normal(size=(m, m))
                Q, R = Mq @ Mq.T + 0.3 * np.eye(n), Mr @ Mr.T + 0.2 * np.eye(m)
            F = random_polytope(rng, m, p, 0.15, 0.45)
            S = 12
            x0 = rng.normal(size=(n, S)) * rng.uniform(0.2, 1.5)
            dA = rng.uniform(-0.03, 0.03, size=(n * n, S)); dB = rng.uniform(-0.03, 0.03, size=(n * m, S))
            sol = hm.mpc(0, A, B, Q, R, Q, None, None, dA, dB, N, x0_soa=x0, F_u=F)
            assert not np.any(sol["flags"] & ~2)
            for s in range(S):
                u, V, act = o.mpc_solve(N, A + dA[:, s].reshape(n, n), B + dB[:, s].reshape(n, m), Q, R, Q, None, None,
                                        x0[:, s], F_u=F)
                assert abs(sol["V"][0, s] - V) < TOL * abs(V) and np.max(np.abs(sol["u0"][0, :, s] - u)) < 1e-9
                n_act += int(act); tot += 1
    assert tot // 4 < n_act < tot
    for n, m in [(2, 1), (3, 2), (4, 2), (3, 3)]:                       # a box handed over as a polytope
        N = 6
        A = rng.normal(size=(n, n)); A *= 1.1 / np.max(np.abs(np.linalg.eigvals(A))); B = rng.normal(size=(n, m))
        Q, R = np.eye(n), 0.5 * np.eye(m)
        lo, hi = -rng.uniform(0.1, 0.4, m), rng.uniform(0.1, 0.4, m)
        F = np.vstack((np.diag(1 / hi), np.diag(1 / lo)))
        S = 24
        x0 = rng.normal(size=(n, S)); dA = rng.uniform(-.02, .02, size=(n * n, S)); dB = rng.uniform(-.02, .02, size=(n * m, S))
        a = hm.mpc(1, A, B, Q, R, Q, lo, hi, dA, dB, N, T=8, x0_soa=x0)
        b = hm.mpc(1, A, B, Q, R, Q, None, None, dA, dB, N, T=8, x0_soa=x0, F_u=F)
        assert relerr(b["J_T"], a["J_T"]) < 1e-12 and np.max(np.abs(a["U"] - b["U"])) < 1e-12
        assert np.array_equal(a["flags"], b["flags"]) and np.any(a["flags"] & 2)
    F = np.array([[1, 0], [0, 1], [-1, 0], [0, -1], [0.5, 0.5], [1, 0], [0.25, 0.25]]) / 0.3
    n, m, N, S = 3, 2, 7, 24
    A = rng.normal(size=(n, n)); A *= 1.15 / np.max(np.abs(np.linalg.eigvals(A))); B = rng.normal(size=(n, m))
    Q, R = 2 * np.eye(n), np.eye(m)
    x0 = rng.normal(size=(n, S)) * 1.5
    z = np.zeros
    xr, ur = rng.normal(size=(n, N)) * 0.2, rng.normal(size=(m, N)) * 0.1
    for refs in ((None, None), (xr, ur)):
        sol = hm.mpc(0, A, B, Q, R, Q, None, None, z((n * n, S)), z((n * m, S)), N, x0_soa=x0, F_u=F, x_ref=refs[0],
                     u_ref=refs[1])
        assert not np.any(sol["flags"] & ~2)
        for s in range(S):
            u, V, _ = o.mpc_solve(N, A, B, Q, R, Q, None, None, x0[:, s], F_u=F, x_ref=refs[0], u_ref=refs[1])
            assert abs(sol["V"][0, s] - V) < TOL * abs(V) and np.max(np.abs(sol["u0"][0, :, s] - u)) < 1e-9


def _golden_inputs(golden, rows):
    eA = np.ascontiguousarray(golden["error_A_f"][:, :, rows, :]).reshape(4, -1)
    eB = np.ascontiguousarray(golden["error_B_f"][:, :, rows, :]).reshape(2, -1)
    return eA, eB


def test_k2_k3_math_reproduce_golden_error_tables(golden, example, known):
    """True cost (K2 simulate), M_V (K2 solve over the ring) and alpha/beta/xi/bound (K3) for 12 systems x 10 levels."""
    rows = slice(0, 12)
    A, B, Q, R, lo, hi = (example[x] for x in ("A", "B", "Q", "R", "lo", "hi"))
    eA, eB = _golden_inputs(golden, rows)
    ring = np.array(known["single"]["x0_vec"])                        # (2, 8): circle_generator(8, 1.5, eps_lqr, Q)
    x_start = ring[:, 1]
    S = eA.shape[1]
    sim = hm.mpc(1, A, B, Q, R, Q, lo, hi, eA, eB, 7, T=30, pts=x_start[None])
    assert relerr(sim["J_T"].reshape(12, 10), golden["true_cost_error"][rows]) < TOL
    mv = hm.mpc(0, A, B, Q, R, Q, lo, hi, eA, eB, 7, pts=ring.T)["M_V"]
    e_per = np.tile(golden["error"], 12)
    b = hm.bounds(A, B, Q, R, lo, hi, eA, eB, 7, e_per, e_per, mv, np.repeat(x_start[:, None], S, axis=1), None,
                  example["p"], float(golden["V_expert"]))
    for k, gk in (("alpha", "alpha_table_error"), ("beta", "beta_table_error"), ("xi", "xi_table_error"),
                  ("bound", "bound_table_error")):
        assert relerr(b[k].reshape(12, 10), golden[gk][rows]) < TOL, k


def test_k3_math_horizon_tables_and_single_example(golden, example, known):
    A, B, Q, R, lo, hi = (example[x] for x in ("A", "B", "Q", "R", "lo", "hi"))
    ring = np.array(known["single"]["x0_vec"]); x_start = ring[:, 1]
    rows = slice(0, 6)
    eA = np.ascontiguousarray(golden["error_A_f"][:, :, rows, 4]).reshape(4, -1)     # level index 4 (utils_class.py:880)
    eB = np.ascontiguousarray(golden["error_B_f"][:, :, rows, 4]).reshape(2, -1)
    S = eA.shape[1]
    for col, N in enumerate(golden["horizon"]):
        N = int(N)
        mv = hm.mpc(0, A, B, Q, R, Q, lo, hi, eA, eB, N, pts=ring.T)["M_V"]
        e = np.full(S, 5e-3)
        b = hm.bounds(A, B, Q, R, lo, hi, eA, eB, N, e, e, mv, np.repeat(x_start[:, None], S, axis=1), None,
                      example["p"], float(golden["V_expert"]))
        for k, gk in (("alpha", "alpha_table_horizon"), ("beta", "beta_table_horizon"), ("xi", "xi_table_horizon"),
                      ("bound", "bound_table_horizon")):
            assert relerr(b[k], golden[gk][rows, col]) < TOL, (k, N)
        sim = hm.mpc(1, A, B, Q, R, Q, lo, hi, eA, eB, N, T=30, pts=x_start[None])
        assert relerr(sim["J_T"], golden["true_cost_horizon"][rows, col]) < TOL
    # working_example_single.py: every intermediate the script prints (zero perturbation, N=6, e=0.01, x = ring[:,0])
    ks = known["single"]
    z4, z2 = np.zeros((4, 1)), np.zeros((2, 1))
    b = hm.bounds(A, B, Q, R, lo, hi, z4, z2, 6, np.array([0.01]), np.array([0.01]), np.array([ks["M_V"]]),
                  ring[:, :1].copy(), None, example["p"], 0.2)
    for key, ref in (("C_K", ks["ex"]["C_K"]), ("rho_K", ks["ex"]["rho_K"]), ("gamma", ks["ex"]["gamma"]),
                     ("rho_gamma", ks["ex"]["rho_gamma"]), ("L_V", ks["bar"]["L_V"]), ("N_0", ks["bar"]["N_0"]),
                     ("omega_N1", ks["omega_eta"]["omega_N1"]), ("omega_N0d5", ks["omega_eta"]["omega_N0d5"]),
                     ("eta", ks["omega_eta"]["eta"]), ("err_th", ks["omega_eta"]["err_th"]),
                     ("N_min", ks["omega_eta"]["N_min"]), ("xi", ks["decrease"]["xi"]),
                     ("alpha", ks["bound"]["alpha"]), ("beta", ks["bound"]["beta"]), ("E_psi", ks["E"]["E_psi"]),
                     ("E_u", ks["E"]["E_u"]), ("E_psi_u", ks["E"]["E_psi_u"]), ("theta_u", ks["theta"]["theta_u"]),
                     ("theta_x_u", ks["theta"]["theta_x_u"]), ("epsilon_K", ks["epsilon_lqr"]),
                     ("bar_u", ks["bar_u"]), ("bar_d_u", ks["bar_d_u"])):
        assert abs(b[key][0] - ref) <= TOL * abs(ref), (key, b[key][0], ref)
    assert relerr(-b["K"][:, 0], np.array(ks["K_lqr"]).ravel()) < TOL          # u = +Kx convention: K = -K_dlqr
    assert relerr(b["P"][:, 0].reshape(2, 2), ks["P_lqr"]) < TOL


def test_k3_math_vs_oracle_multi_input():
    """m > 1 (where the reference itself raises, utils.py:356): the oracle restatement is the yardstick."""
    for n, m, N in [(4, 2, 10), (3, 2, 6), (2, 2, 4)]:
        A, B, Q, R = nb.synth_problem(n, m, seed=2)
        Q = 1.5 * Q
        lo, hi = -0.3 * np.ones(m), 0.4 * np.ones(m)
        dA, dB, x0 = nb.synth_samples(n, m, 6, seed=4, e=0.01)
        sA, sB, sx = nb.to_soa(dA, dB, x0)
        e = np.full(6, 0.01); mv = np.linspace(0.5, 2.0, 6)
        p = np.array([0.1, 1, 0.6])
        b = hm.bounds(A, B, Q, R, lo, hi, sA, sB, N, e, e, mv, sx, None, p, 1.0)
        for s in range(6):
            Ah, Bh = A + dA[s], B + dB[s]
            K, _ = o.dlqr(Ah, Bh, Q, R)
            try:
                dec = o.energy_decreasing(Ah, Bh, Q, R, lo, hi, N, 0.01, 0.01, -K, mv[s])
            except ValueError:
                assert b["flags"][s] & 512
                continue
            bnd = o.energy_bound(Ah, Bh, Q, R, lo, hi, N, 0.01, 0.01, x0[s], p)
            for key, ref in (("xi", dec["xi"]), ("eta", dec["eta"]), ("alpha", bnd["alpha"]), ("beta", bnd["beta"])):
                assert abs(b[key][s] - ref) <= TOL * abs(ref), (n, m, key)


def test_k3_math_unit_norm_branch_of_geo_M():
    """geo_M's exact-equality branch `norm == 1` (utils.py:404-405): for ||A||_2 == 1.0 the geometric sum is N - 1, not
    (1 - f^(2N-2)) / (1 - f^2) = 0 / 0. A = diag(1, 0.3) has the 2-norm exactly 1 in LAPACK and in the engine's Jacobi
    norm alike; a neighbour 1 - 2^-30 takes the other branch. Both must match the oracle."""
    for a11 in (1.0, 1.0 - 2.0 ** -30):
        A = np.diag([a11, 0.3]); B = np.array([[1.0], [0.5]]); Q = 2 * np.eye(2); R = np.eye(1)
        lo, hi = np.array([-0.1]), np.array([0.1])
        N = 7
        z = np.zeros
        x = np.array([[0.05], [0.02]])
        K = -o.dlqr(A, B, Q, R)[0]
        b = hm.bounds(A, B, Q, R, lo, hi, z((4, 1)), z((2, 1)), N, np.array([5e-3]), np.array([5e-3]),
                      np.array([0.05]), x, K.reshape(-1, 1), np.array([0.1, 1, 0.6]), 0.2)
        assert (b["norm_A"][0] == 1.0) == (a11 == 1.0)
        dec = o.energy_decreasing(A, B, Q, R, lo, hi, N, 5e-3, 5e-3, K, 0.05)
        for key in ("xi", "eta", "omega_N1", "omega_N0d5"):
            assert abs(b[key][0] - dec[key]) <= TOL * abs(dec[key]), (a11, key)


def test_k3_sturm_search_vs_lapack():
    """K3's search for both extremes of a symmetric tridiagonal (three shifts per search and pass) vs LAPACK on random,
    Toeplitz (clustered ends), identity, graded, tightly clustered, 16-decade and split matrices, k = 1..78."""
    import scipy.linalg as sla
    rng = np.random.default_rng(0)

    def check(d, e):
        k = len(d)
        ev = sla.eigvalsh_tridiagonal(d, e[1:]) if k > 1 else np.array(d)
        lo, hi = hm.tridiag_extremes(d, e)
        nrm = max(abs(ev[0]), abs(ev[-1]), 1e-300)
        assert max(abs(lo - ev[0]), abs(hi - ev[-1])) <= 5e-15 * nrm

    check(np.array([3.5]), np.zeros(1))
    for k in (2, 3, 4, 5, 8, 13, 20, 36, 50, 64, 78):
        for _ in range(20):
            check(rng.normal(size=k) * rng.uniform(0.1, 10),
                  np.concatenate(([0], rng.normal(size=k - 1) * rng.uniform(0.01, 5))))
        check(2 * np.ones(k), np.concatenate(([0], -np.ones(k - 1))))
        check(np.ones(k), np.zeros(k))
        check(np.arange(k, dtype=float), np.concatenate(([0], np.full(k - 1, 1e-8))))
        check(np.ones(k), np.concatenate(([0], np.full(k - 1, 1e-9))))
        d = 10.0 ** rng.uniform(-8, 8, size=k)
        check(d, np.concatenate(([0], np.sqrt(d[:-1] * d[1:]) * rng.uniform(0, 0.5, k - 1))))
        e = np.full(k, 0.3); e[0] = 0.0; e[k // 2] = 0.0
        check(np.concatenate((np.ones(k // 2), 5 * np.ones(k - k // 2))), e)


def test_k2_math_long_horizon_late_saturation_vs_dense_qp():
    """Round 2: the unconstrained cost-to-go is kept for the first 12 stages only and the stage loops run one stage ahead
    of their loads. Long horizons whose inputs saturate LATE (working set beyond stage 12 -> the full N-stage sweep) and
    early (-> restart from the stored S_k), marginally unstable plants, both vs the dense Cholesky + BVLS oracle; the
    closed loop (certificate fast path with the register-held stage-0 gain) vs the same oracle stepped on the host."""
    from oracle import np_oracle as o
    rng = np.random.default_rng(2024)
    late = early = 0
    for (n, m) in [(2, 1), (2, 2), (3, 1), (4, 2)]:
        for rep in range(3):
            N = int(rng.integers(20, 41))
            A = rng.normal(size=(n, n))
            A *= rng.uniform(0.95, 1.15) / np.max(np.abs(np.linalg.eigvals(A)))
            B = rng.normal(size=(n, m))
            Q = rng.uniform(0.5, 3) * np.eye(n); R = rng.uniform(0.1, 2) * np.eye(m)
            lo, hi = -rng.uniform(0.02, 0.1, size=m), rng.uniform(0.02, 0.1, size=m)
            S = 6
            x0 = rng.normal(size=(n, S)) * rng.uniform(0.5, 3.0)
            sol = hm.mpc(0, A, B, Q, R, Q, lo, hi, None, None, N, x0_soa=x0)
            assert not np.any(sol["flags"] & ~2)
            for s in range(S):
                ur, Vr, _ = o.mpc_solve(N, A, B, Q, R, Q, lo, hi, x0[:, s], exact_fast=False)
                assert abs(sol["V"][0, s] - Vr) < TOL * abs(Vr), (n, m, N, s)
                assert np.max(np.abs(sol["u0"][0, :, s] - ur)) < TOL, (n, m, N, s)
                H, gq, _ = o.condensed_qp(N, A, B, Q, R, Q, x0[:, s])
                z = o.box_qp(H, gq, np.tile(lo, N), np.tile(hi, N)).reshape(N, m)
                sat = np.flatnonzero(np.any((z <= lo + 1e-12) | (z >= hi - 1e-12), axis=1))
                if sat.size:
                    late += int(sat.max() >= 12)
                    early += int(sat.max() < 12)
    assert late >= 10 and early >= 1, (late, early)      # both restart routes were taken
    # closed loop: T steps of the exact QP on the true plant (= model here), first steps saturated, later ones certified
    A = np.array([[1, 0.7], [0.12, 0.4]]); B = np.array([[1], [1.2]])
    Q = 2 * np.eye(2); R = np.eye(1); lo, hi = np.array([-0.1]), np.array([0.1])
    x0 = np.array([[0.3], [0.25]])
    N, T = 25, 30
    sim = hm.mpc(1, A, B, Q, R, Q, lo, hi, None, None, N, T=T, x0_soa=x0)
    x = x0[:, 0].copy()
    J = float(x @ Q @ x)
    for t in range(T):
        u, _, _ = o.mpc_solve(N, A, B, Q, R, Q, lo, hi, x, exact_fast=False)
        assert np.max(np.abs(sim["U"][t, :, 0] - u)) < 1e-9, t
        x = A @ x + B @ u
        J += float(x @ Q @ x + u @ R @ u)
    assert abs(sim["J_T"][0] - J) < TOL * J


def _scale_to_saturation(Ah, Bh, Q, R, N, lo, hi, X, t):
    """Columns of X rescaled so that the unconstrained plan of model s from column s peaks at t[s] times the input box:
    t > 1 makes the box active, t < 1 leaves the plan feasible (the plan is linear in the initial state)."""
    out = X.copy()
    for s in range(X.shape[1]):
        K, _ = o.riccati(Ah[s], Bh[s], Q, R, Q, N)
        x, r = X[:, s], 0.0
        for k in range(N):
            u = K[k] @ x
            r = max(r, float(np.max(np.maximum(u / hi, u / lo))))
            x = Ah[s] @ x + Bh[s] @ u
        out[:, s] *= t[s] / r
    return out


@pytest.mark.parametrize("n,m", COMPILED_DIMS)
def test_k2_math_every_compiled_pair_vs_dense_qp(n, m):
    """Box solve and closed loop of every compiled (n, m) — (1, 1), (3, 3) and (4, 4) included, the last two being the
    n <= 4 pairs that re-read the stage-0 gain from scratch on the certificate path — vs the dense Cholesky + BVLS
    oracle: a short horizon (the whole cost-to-go stored) and a long one (20..40 stages) with general SPD weights, model
    != plant, most initial states saturating and some not; the closed loop runs until the certificate takes over."""
    rng = np.random.default_rng(40 + 10 * n + m)
    S, T = 6, 30
    for N, general in ((int(rng.integers(3, 12)), False), (int(rng.integers(20, min(40, 256 // m) + 1)), True)):
        A = rng.normal(size=(n, n)); A *= rng.uniform(0.6, 1.0) / np.max(np.abs(np.linalg.eigvals(A)))
        B = rng.normal(size=(n, m))
        if general:
            Mq, Mr = rng.normal(size=(n, n)), rng.normal(size=(m, m))
            Q, R = Mq @ Mq.T / n + 0.5 * np.eye(n), Mr @ Mr.T / m + 0.3 * np.eye(m)
        else:
            Q, R = rng.uniform(0.5, 3) * np.eye(n), rng.uniform(0.1, 2) * np.eye(m)
        lo, hi = -rng.uniform(0.05, 0.4, size=m), rng.uniform(0.05, 0.4, size=m)
        dA = rng.uniform(-0.01, 0.01, size=(n * n, S)); dB = rng.uniform(-0.01, 0.01, size=(n * m, S))
        Ah = [A + dA[:, s].reshape(n, n) for s in range(S)]
        Bh = [B + dB[:, s].reshape(n, m) for s in range(S)]
        t = np.r_[rng.uniform(0.2, 0.8, 2), rng.uniform(1.2, 3.0, S - 2)]
        x0 = _scale_to_saturation(Ah, Bh, Q, R, N, lo, hi, rng.normal(size=(n, S)), t)
        sol = hm.mpc(0, A, B, Q, R, Q, lo, hi, dA, dB, N, x0_soa=x0)
        sim = hm.mpc(1, A, B, Q, R, Q, lo, hi, dA, dB, N, T=T, x0_soa=x0)
        assert not np.any(sol["flags"] & ~2) and not np.any(sim["flags"] & ~2)
        certified = 0
        for s in range(S):
            ur, Vr, act = o.mpc_solve(N, Ah[s], Bh[s], Q, R, Q, lo, hi, x0[:, s])
            assert act == (t[s] > 1) and bool(sol["flags"][0, s] & 2) == act, (n, m, N, s)
            if not act:
                ur, Vr, _ = o.mpc_solve(N, Ah[s], Bh[s], Q, R, Q, lo, hi, x0[:, s], exact_fast=False)
            assert abs(sol["V"][0, s] - Vr) < TOL * abs(Vr), (n, m, N, s)
            assert np.max(np.abs(sol["u0"][0, :, s] - ur)) < TOL, (n, m, N, s)
            so = o.simulate(T, N, Ah[s], Bh[s], Q, R, Q, lo, hi, x0[:, s], A, B)
            assert abs(sim["J_T"][s] - so["J_T"]) < TOL * so["J_T"], (n, m, N, s)
            assert np.max(np.abs(sim["U"][:, :, s].T - so["U"])) < TOL, (n, m, N, s)
            assert np.max(np.abs(sim["X"][:, :, s].T - so["X"])) < TOL * max(1.0, np.max(np.abs(so["X"])))
            assert sim["n_active"][s] == so["n_active"], (n, m, N, s)
            certified += int(so["n_active"] < T - 5)
        assert certified >= S // 2, (n, m, N)          # the later steps of most closed loops are unconstrained
