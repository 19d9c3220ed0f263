"""GPU parity tests (run on the B200 box: `pytest -m gpu`). Everything goes through the C ABI
(lq_mpc_b200.engine -> liblqmpc_b200.so) or through the drop-in classes on top of it, and is compared with
  * the reference's shipped golden file and the answers generated from the untouched reference (tests/golden/),
  * the CPU oracle (oracle/np_oracle.py, oracle/np_batched.py) on the same seeded inputs.
Tolerance: 1e-9 relative (BASELINE.json north_star) unless a test states a tighter one. Where the engine and the
float64 oracle differ by more than that, NEITHER is trusted: tests/mp_truth.py recomputes the quantity in 50-digit
arithmetic and the engine must be within 1e-9 of THAT (or within the stated, computed condition bound).
"""
import math
import os

import numpy as np
import pytest

from tests.conftest import relerr

pytestmark = pytest.mark.gpu
TOL = 1e-9


def _soa(dA, dB, x0):
    from oracle import np_batched as nb
    return nb.to_soa(dA, dB, x0)


def _k1_arbitrate(A, B, Q, R, dA, dB, x0, N_min, got_J, ref_J, ref_rho, max_cases=12):
    """Entries where engine and oracle disagree on J_inf by more than 1e-9 (only possible next to the stability
    boundary, where J ~ 1/(1 - rho) is ill-conditioned): both are measured against the 50-digit value; the engine must
    be within max(1e-9, 16 u rho / (1 - rho)) of it (mp_truth.j_condition_bound)."""
    from tests import mp_truth as mt
    fin = np.isfinite(ref_J) & np.isfinite(got_J)
    err = np.where(fin, np.abs(got_J - ref_J) / np.where(fin, np.abs(ref_J), 1.0), 0.0)
    bad = np.argwhere(err > TOL)
    assert len(bad) <= max_cases, "engine and oracle disagree beyond 1e-9 on %d entries" % len(bad)
    for h, s in bad:
        t = mt.k1_truth(A, B, Q, R, Q, dA[s], dB[s], x0[s], N_min + h)
        assert abs(got_J[h, s] - t["J"]) <= mt.j_condition_bound(t["rho"]) * abs(t["J"]), (h, s, t["rho"])
        assert 1.0 - ref_rho[h, s] < 2e-6, "disagreement away from the stability boundary"
    return len(bad)


# ------------------------------------------------------------------------------------------------------- K1
@pytest.mark.parametrize("n,m,e", [(4, 2, 0.01), (2, 1, 0.05), (1, 1, 0.1), (3, 2, 0.3), (3, 3, 0.1), (4, 1, 0.05),
                                   (4, 4, 0.2), (6, 2, 0.05), (8, 2, 0.02), (2, 2, 0.1), (3, 1, 0.1)])
def test_k1_matches_oracle(engine, n, m, e):
    from oracle import np_batched as nb
    A, B, Q, R = nb.synth_problem(n, m, seed=0)
    engine.set_problem(A, B, Q, R, Q, None, None, 30)
    S = 4099                                            # ragged: not a multiple of the block size
    dA, dB, x0 = nb.synth_samples(n, m, S, seed=1, e=e)
    Pexp = nb.expert_matrix(A, B, Q, R, Q, 30)
    ref = nb.eval_batch(A, B, Q, R, Q, Pexp, dA, dB, x0, 2, 11, T=25, want_K=True)
    got = engine.eval_batch(*_soa(dA, dB, x0), 2, 11, T=25, want=("J", "rho", "ratio", "flags", "V_N", "J_T", "K0"))
    g = {k: v.cpu().numpy() for k, v in got.items() if hasattr(v, "cpu")}
    assert relerr(engine.prepared()["Pexp"], Pexp) < 1e-12
    assert np.array_equal((g["flags"] & 1) != 0, ref["unstable"])
    for k, kr in (("rho", "rho"), ("V_N", "Vn"), ("J_T", "JT")):
        assert relerr(g[k], ref[kr]) < TOL, k
    # J_inf, ratio: 1e-9 on EVERY entry; an entry that misses it is arbitrated in 50-digit arithmetic (J ~ 1/(1 - rho)
    # is ill-conditioned within ~2e-6 of the stability boundary — n = m = 1, e = 0.1 has a few such samples)
    n_arb = _k1_arbitrate(A, B, Q, R, dA, dB, x0, 2, g["J"], ref["J"], ref["rho"])
    assert np.array_equal(np.isfinite(g["J"]), np.isfinite(ref["J"]))
    fin = np.isfinite(ref["J"])
    assert np.max(np.abs(g["ratio"][fin] / g["J"][fin] - ref["ratio"][fin] / ref["J"][fin])
                  * np.abs(ref["J"][fin] / ref["ratio"][fin])) < TOL      # ratio = J / V_expert: same V_expert
    assert n_arb == 0 or (n, m) == (1, 1)
    K = g["K0"].reshape(10, m, n, S).transpose(0, 3, 1, 2)
    assert np.max(np.abs(K - ref["K0"])) < 1e-10 * max(1.0, np.max(np.abs(ref["K0"])))
    assert not np.any(g["flags"] & ~1)


@pytest.mark.parametrize("n,m,variant", [(8, 2, ""), (8, 2, "0"), (6, 2, ""), (6, 2, "0")])
def test_k1_lane_group_builds_agree_with_thread_route_and_oracle(engine, n, m, variant, monkeypatch):
    """n = 6, 8: the lane-group kernel (k_group.cu; default) and the thread-per-sample instantiation
    (LQMPC_K1_GROUP=0) against the oracle — one horizon per sample (the build whose
    cost-to-go dies before the closed-loop phase) and nested horizons (the build that parks it in shared memory),
    a ragged batch (tail groups), large perturbations (unstable closed loops) included."""
    from oracle import np_batched as nb
    if variant:
        monkeypatch.setenv("LQMPC_K1_GROUP", variant)
    else:
        monkeypatch.delenv("LQMPC_K1_GROUP", raising=False)
    A, B, Q, R = nb.synth_problem(n, m, seed=2)
    engine.set_problem(A, B, Q, R, Q, None, None, 30)
    Pexp = nb.expert_matrix(A, B, Q, R, Q, 30)
    for S, e, (N_min, N_max) in ((1031, 0.05, (7, 7)), (517, 0.4, (1, 5)), (3, 0.02, (1, 1))):
        dA, dB, x0 = nb.synth_samples(n, m, S, seed=11 + S, e=e)
        ref = nb.eval_batch(A, B, Q, R, Q, Pexp, dA, dB, x0, N_min, N_max, T=0, want_K=True)
        want = ("J", "rho", "ratio", "flags", "K0") + (("V_N",) if N_min != N_max else ())
        got = engine.eval_batch(*_soa(dA, dB, x0), N_min, N_max, want=want)
        g = {k: v.cpu().numpy() for k, v in got.items() if hasattr(v, "cpu")}
        assert np.array_equal((g["flags"] & 1) != 0, ref["unstable"]), (S, e)
        assert not np.any(g["flags"] & ~1)
        assert relerr(g["rho"], ref["rho"]) < TOL
        if "V_N" in g:
            assert relerr(g["V_N"], ref["Vn"]) < TOL
        _k1_arbitrate(A, B, Q, R, dA, dB, x0, N_min, g["J"], ref["J"], ref["rho"])
        assert np.array_equal(np.isfinite(g["J"]), np.isfinite(ref["J"]))
        H = N_max - N_min + 1
        K = g["K0"].reshape(H, m, n, S).transpose(0, 3, 1, 2)
        assert np.max(np.abs(K - ref["K0"])) < 1e-10 * max(1.0, np.max(np.abs(ref["K0"])))


def test_k1_lane_group_spectral_radius_on_hard_spectra(engine):
    """The lane-group kernel takes rho from repeated squaring with a dominant-pair early acceptance (k_group.cu). With
    a vanishing input matrix the closed loop IS the plant, so prescribed spectra reach that code: a dominant real
    eigenvalue, a +- pair, a complex pair, three eigenvalues of (nearly) equal modulus, a defective (Jordan) dominant
    eigenvalue, a nilpotent plant. Compared with numpy's eigenvalues; where the two differ by more than 1e-9 the
    dominant eigenvalue is ill-conditioned and both must lie within its condition bound of the 50-digit value."""
    import mpmath as mp
    rng = np.random.default_rng(77)
    n, m = 8, 2

    def from_spec(spec, V):
        D = np.zeros((n, n)); i = 0
        for sp_ in spec:
            if sp_[0] == "c":
                a, b = sp_[1] * np.cos(sp_[2]), sp_[1] * np.sin(sp_[2])
                D[i:i + 2, i:i + 2] = [[a, b], [-b, a]]; i += 2
            elif sp_[0] == "j":                        # Jordan block of size 3
                for q in range(3):
                    D[i + q, i + q] = sp_[1]
                D[i, i + 1] = D[i + 1, i + 2] = 1.0; i += 3
            else:
                D[i, i] = sp_[1]; i += 1
        while i < n:
            D[i, i] = rng.uniform(-0.4, 0.4) * abs(spec[0][1]); i += 1
        return V @ D @ np.linalg.inv(V)

    mats = []
    for t in range(60):
        V = rng.standard_normal((n, n))
        r0 = rng.uniform(0.3, 1.3)
        gap = 10.0 ** rng.uniform(-12, -1)
        th, th2 = rng.uniform(0.05, 3.0, 2)
        kind = t % 6
        if kind == 0: spec = [("r", r0)]
        elif kind == 1: spec = [("r", r0), ("r", -r0 * (1 - gap))]
        elif kind == 2: spec = [("c", r0, th)]
        elif kind == 3: spec = [("c", r0, th), ("r", r0 * (1 - gap)), ("c", r0 * (1 - 3 * gap), th2)]
        elif kind == 4: spec = [("j", r0)]
        else: spec = [("r", r0), ("r", r0 * (1 - gap)), ("r", -r0 * (1 - 2 * gap))]
        mats.append(from_spec(spec, V))
    N8 = np.zeros((n, n)); N8[np.arange(n - 1), np.arange(1, n)] = rng.uniform(0.5, 2.0, n - 1)
    mats.append(N8)                                     # nilpotent: rho = 0
    mats.append(np.zeros((n, n)))
    mp.mp.dps = 50
    n_arb = 0
    for M in mats:
        B = np.zeros((n, m)); B[0, 0] = B[1, 1] = 1e-200          # K = O(1e-200): A + B K == A in double
        engine.set_problem(M, B, np.eye(n), np.eye(m), np.eye(n), None, None, 1)
        z = np.zeros((1, n, n)), np.zeros((1, n, m)), np.ones((1, n))
        got = engine.eval_batch(*_soa(*z), 1, 1, want=("rho", "flags"))
        rho = float(got["rho"].cpu().numpy()[0, 0])
        ref = float(np.max(np.abs(np.linalg.eigvals(M))))
        if abs(rho - ref) <= TOL * max(ref, 1e-300) or (ref < 1e-12 and rho < 1e-12):
            continue
        n_arb += 1
        ev = mp.eig(mp.matrix(M.tolist()), left=False, right=False)
        truth = float(max(abs(x) for x in ev))
        w, vl, vr = __import__("scipy.linalg", fromlist=["eig"]).eig(M, left=True)
        j = int(np.argmax(np.abs(w)))
        kappa = np.linalg.norm(vl[:, j]) * np.linalg.norm(vr[:, j]) / abs(np.vdot(vl[:, j], vr[:, j]))
        bound = max(TOL, 64 * np.finfo(float).eps * kappa * np.linalg.norm(M, 2) / truth)
        assert abs(rho - truth) <= bound * truth, (rho, truth, ref, kappa)
    assert n_arb <= 25


def test_k1_per_sample_oracle_and_edges(engine):
    """Independent per-sample oracle (scipy Lyapunov/eig) + edge cases: S=1, S=0, N=1, nested == single horizon."""
    from oracle import np_batched as nb, np_oracle as o
    A, B, Q, R = nb.synth_problem(4, 2, seed=3)
    engine.set_problem(A, B, Q, R, Q, None, None, 0)          # N_opc <= 0: DARE limit for the expert cost
    P_inf = o.dlqr(A, B, Q, R)[1]
    assert relerr(engine.prepared()["Pexp"], P_inf) < 1e-10
    dA, dB, x0 = nb.synth_samples(4, 2, 64, seed=5, e=0.05)
    got = engine.eval_batch(*_soa(dA, dB, x0), 1, 6, want=("J", "rho", "ratio", "flags"))
    J, rho, ratio = (got[k].cpu().numpy() for k in ("J", "rho", "ratio"))
    for s in range(0, 64, 7):
        for N in (1, 3, 6):
            K = o.riccati(A + dA[s], B + dB[s], Q, R, Q, N)[0][0]
            Jr, rr = o.closed_loop_inf_cost(A, B, K, Q, R, x0[s])
            assert abs(rho[N - 1, s] - rr) <= TOL * rr
            if math.isinf(Jr):
                assert math.isinf(J[N - 1, s]) and math.isinf(ratio[N - 1, s])
                continue
            assert abs(J[N - 1, s] - Jr) <= TOL * abs(Jr)
            assert abs(ratio[N - 1, s] - Jr / (x0[s] @ P_inf @ x0[s])) <= TOL * ratio[N - 1, s]
    one = engine.eval_batch(*_soa(dA[:1], dB[:1], x0[:1]), 6, 6)
    assert one["J"].shape == (1, 1) and float(one["J"][0, 0]) == J[5, 0]         # nested == single, bit for bit
    empty = engine.eval_batch(np.zeros((16, 0)), np.zeros((8, 0)), np.zeros((4, 0)), 1, 2)
    assert empty["J"].shape == (2, 0)


def test_k1_cfg4_vs_untouched_reference(engine, cfg4):
    """BASELINE configs[3] shape (n = 4, m = 2, N = 10) pinned on the reference ITSELF: twelve samples that went
    through the untouched LQ_MPC_Controller / LQ_MPC_Simulator (utils_class.py:48-91, 245-285; loose input box, so the
    cvxpy problem is the unconstrained one; T = 400). K1's first-step gain, V_N, J_T(400) and J_inf vs those answers,
    and the exact-QP kernels (K2) on the same samples."""
    A, B = np.array(cfg4["A"]), np.array(cfg4["B"])
    n, m, N, T = cfg4["n"], cfg4["m"], cfg4["N"], cfg4["T"]
    cs = cfg4["cases"]
    dA = np.array([c["dA"] for c in cs]); dB = np.array([c["dB"] for c in cs]); x0 = np.array([c["x0"] for c in cs])
    engine.set_problem(A, B, np.eye(n), np.eye(m), np.eye(n), None, None, 30)
    got = engine.eval_batch(*_soa(dA, dB, x0), N, N, T=T, want=("J", "rho", "V_N", "J_T", "K0", "flags"))
    g = {k: v.cpu().numpy() for k, v in got.items() if hasattr(v, "cpu")}
    assert not g["flags"].any()
    for s, c in enumerate(cs):
        K = g["K0"][0, :, s].reshape(m, n)
        assert np.max(np.abs(K - np.array(c["K0"]))) < 1e-10 * max(1.0, np.max(np.abs(K)))
        assert abs(g["J_T"][0, s] - c["J_T"]) <= TOL * c["J_T"]                # finite sum, reference semantics
        assert abs(g["J"][0, s] - c["J_T"]) <= TOL * c["J_T"]                  # Lyapunov limit == J_T(400) to rounding
        assert abs(g["V_N"][0, s] - c["V_N"]) <= TOL * c["V_N"]
        assert g["rho"][0, s] < 1.0
    engine.set_problem(A, B, np.eye(n), np.eye(m), np.eye(n), -1e6 * np.ones(m), 1e6 * np.ones(m), 30)
    sa, sb, sx = _soa(dA, dB, x0)
    sol = engine.mpc_solve_batch(sa, sb, N, x0=sx)
    sim = engine.simulate_batch(sa, sb, N, T, x0=sx, want=("J_T", "X", "U", "flags"))
    assert not sol["flags"].cpu().numpy().any() and not sim["flags"].cpu().numpy().any()
    for s, c in enumerate(cs):
        assert abs(float(sol["V"][0, s]) - c["V_N"]) <= TOL * c["V_N"]
        assert np.max(np.abs(sol["u0"].cpu().numpy()[0, :, s] - np.array(c["u_0"]))) < 1e-10
        assert abs(float(sim["J_T"][s]) - c["J_T"]) <= TOL * c["J_T"]
        assert np.max(np.abs(sim["U"].cpu().numpy()[:5, :, s].T - np.array(c["U_head"]))) < 1e-10


def test_k1_seeded_entry_point(engine):
    """lqmpc_eval_seeded: (dA, dB, x0) drawn INSIDE the kernel from the global sample index. The tables must equal the
    oracle evaluated on the numpy restatement of the same Philox stream (1e-9; the uniforms are bit-exact), the fused
    column moments must equal numpy on those tables, two shards must reproduce one batch bit for bit, and the
    moments-only call (tables in the context's scratch) must return the same moments."""
    import torch
    from oracle import np_batched as nb, np_sampler as ns
    from lq_mpc_b200 import stats
    A, B, Q, R = nb.synth_problem(4, 2, seed=0)
    engine.set_problem(A, B, Q, R, Q, None, None, 30)
    S, first = 20_001, (1 << 32) - 7000                      # the index range crosses 2^32
    got = engine.eval_seeded(1, first, S, 0.01, 0.01, 9, 10, want=("J", "rho", "ratio", "flags", "moments"))
    dA, dB, x0 = ns.seeded_samples(1, first, S, 4, 2, 0.01, 0.01)
    ref = nb.eval_batch(A, B, Q, R, Q, nb.expert_matrix(A, B, Q, R, Q, 30), dA, dB, x0, 9, 10)
    for k in ("J", "rho", "ratio"):
        assert relerr(got[k].cpu().numpy(), ref[k]) < TOL, k
    assert not got["flags"].cpu().numpy().any()
    tab = got["table"].cpu().numpy()
    st = stats.merge_moments(got["moments"].cpu().numpy()[None])
    assert np.array_equal(st["max"], tab.max(axis=1)) and np.array_equal(st["min"], tab.min(axis=1))
    assert relerr(st["mean"], tab.mean(axis=1)) < 1e-12 and relerr(st["std"], tab.std(axis=1)) < 1e-9
    only = engine.eval_seeded(1, first, S, 0.01, 0.01, 9, 10, want=("moments",))
    assert torch.equal(only["moments"], got["moments"])
    a = engine.eval_seeded(1, first, 12_000, 0.01, 0.01, 9, 10, want=("J", "rho", "ratio"))
    b = engine.eval_seeded(1, first + 12_000, S - 12_000, 0.01, 0.01, 9, 10, want=("J", "rho", "ratio"))
    assert torch.equal(torch.cat([a["table"], b["table"]], dim=1), got["table"])
    # different error levels for A and B, another shape
    A2, B2, Q2, R2 = nb.synth_problem(2, 1, seed=0)
    engine.set_problem(A2, B2, Q2, R2, Q2, None, None, 30)
    g2 = engine.eval_seeded(9, 0, 3001, 0.03, 0.002, 5, 5, want=("J", "rho", "ratio"))
    dA2, dB2, x2 = ns.seeded_samples(9, 0, 3001, 2, 1, 0.03, 0.002)
    r2 = nb.eval_batch(A2, B2, Q2, R2, Q2, nb.expert_matrix(A2, B2, Q2, R2, Q2, 30), dA2, dB2, x2, 5, 5)
    assert relerr(g2["J"].cpu().numpy(), r2["J"]) < TOL and relerr(g2["rho"].cpu().numpy(), r2["rho"]) < TOL
    assert engine.eval_seeded(1, 0, 0, 0.01, 0.01, 3, 3, want=("J",))["J"].shape == (1, 0)


@pytest.mark.parametrize("n,m", [(8, 2), (6, 2)])
def test_k1_seeded_entry_point_on_lane_groups(engine, n, m, monkeypatch):
    """lqmpc_eval_seeded at n = 6, 8: every lane of a group draws its own rows from the (sample, pair)-addressed Philox
    stream. Same checks as above, plus: the lane-group build and the thread-per-sample build (LQMPC_K1_GROUP=0) see the
    same samples (their tables agree to 1e-9; the evaluation arithmetic differs, the operands do not)."""
    import torch
    from oracle import np_batched as nb, np_sampler as ns
    monkeypatch.delenv("LQMPC_K1_GROUP", raising=False)
    A, B, Q, R = nb.synth_problem(n, m, seed=1)
    engine.set_problem(A, B, Q, R, Q, None, None, 30)
    S, first = 5_003, (1 << 32) - 2000
    got = engine.eval_seeded(3, first, S, 0.02, 0.005, 4, 6, want=("J", "rho", "ratio", "flags", "moments"))
    dA, dB, x0 = ns.seeded_samples(3, first, S, n, m, 0.02, 0.005)
    ref = nb.eval_batch(A, B, Q, R, Q, nb.expert_matrix(A, B, Q, R, Q, 30), dA, dB, x0, 4, 6)
    for k in ("J", "rho", "ratio"):
        assert relerr(got[k].cpu().numpy(), ref[k]) < TOL, k
    assert not got["flags"].cpu().numpy().any()
    a = engine.eval_seeded(3, first, 3_000, 0.02, 0.005, 4, 6, want=("J", "rho", "ratio"))
    b = engine.eval_seeded(3, first + 3_000, S - 3_000, 0.02, 0.005, 4, 6, want=("J", "rho", "ratio"))
    assert torch.equal(torch.cat([a["table"], b["table"]], dim=1), got["table"])
    one = engine.eval_seeded(3, first, S, 0.02, 0.005, 6, 6, want=("J", "rho"))       # the one-horizon build
    assert relerr(one["J"].cpu().numpy(), ref["J"][2:3]) < TOL
    monkeypatch.setenv("LQMPC_K1_GROUP", "0")
    thr = engine.eval_seeded(3, first, S, 0.02, 0.005, 4, 6, want=("J", "rho", "ratio"))
    assert relerr(thr["table"].cpu().numpy(), got["table"].cpu().numpy()) < TOL


def test_k1_unstable_flagged(engine):
    """An estimated model far from the plant gives an unstable closed loop: J = +inf, flag bit 0, rho >= 1."""
    A = np.array([[1.2, 0.5], [0.0, 1.1]])
    B = np.array([[0.0], [1.0]])
    engine.set_problem(A, B, np.eye(2), np.eye(1), np.eye(2), None, None, 30)
    dA = np.zeros((4, 2)); dB = np.zeros((2, 2)); x0 = np.ones((2, 2))
    dB[1, 1] = -2.5                                     # controller believes the input gain has the opposite sign
    got = engine.eval_batch(dA, dB, x0, 5, 5)
    J, rho, fl = (got[k].cpu().numpy()[0] for k in ("J", "rho", "flags"))
    assert np.isfinite(J[0]) and fl[0] == 0 and rho[0] < 1
    assert np.isinf(J[1]) and (fl[1] & 1) and rho[1] >= 1


def test_k1_full_size_properties(engine):
    """BASELINE size (1.25e7 samples per GPU): size-independent properties instead of an oracle run.
    J is quadratic in x0 (J(2 x0) = 4 J(x0) exactly in binary FP), rho and ratio do not depend on the scaling,
    the host-buffer pipeline returns exactly the device-resident result, a subsample matches the oracle."""
    import torch
    from lq_mpc_b200 import sampling as sp
    from oracle import np_batched as nb
    S = 12_500_000
    A, B, Q, R = sp.synth_problem(4, 2, seed=0)
    engine.set_problem(A, B, Q, R, Q, None, None, 30)
    g = torch.Generator(device="cuda").manual_seed(7)
    dA = (torch.rand((16, S), device="cuda", dtype=torch.float64, generator=g) - 0.5) * 0.02
    dB = (torch.rand((8, S), device="cuda", dtype=torch.float64, generator=g) - 0.5) * 0.02
    x0 = torch.randn((4, S), device="cuda", dtype=torch.float64, generator=g)
    r1 = engine.eval_batch(dA, dB, x0, 10, 10)
    r2 = engine.eval_batch(dA, dB, 2.0 * x0, 10, 10)
    assert torch.equal(r2["J"], 4.0 * r1["J"])
    assert torch.equal(r2["rho"], r1["rho"])
    assert torch.equal(r2["ratio"], r1["ratio"])
    assert int((r1["flags"] != 0).sum()) == 0
    assert float(r1["ratio"].min()) >= 1.0 - 1e-9       # the expert (N_opc=30, true model) is at least as good ... to 1e-9
    idx = torch.arange(0, S, 9973, device="cuda")
    sub = [t[:, idx].cpu().numpy() for t in (dA, dB, x0)]
    Pexp = nb.expert_matrix(A, B, Q, R, Q, 30)
    ref = nb.eval_batch(A, B, Q, R, Q, Pexp, sub[0].T.reshape(-1, 4, 4), sub[1].T.reshape(-1, 4, 2), sub[2].T, 10, 10)
    assert relerr(r1["J"][:, idx].cpu().numpy(), ref["J"]) < TOL
    assert relerr(r1["rho"][:, idx].cpu().numpy(), ref["rho"]) < TOL
    # host path on a slice (pinned host buffers, chunked pipeline)
    Sh = 1_000_003
    h = [t[:, :Sh].contiguous().cpu().pin_memory() for t in (dA, dB, x0)]
    out = engine.eval_batch_host(h[0], h[1], h[2], 10, 10, chunk=1 << 18)
    assert torch.equal(out["J"], r1["J"][:, :Sh].cpu())
    assert torch.equal(out["ratio"], r1["ratio"][:, :Sh].cpu())
    assert torch.equal(out["flags"], r1["flags"][:, :Sh].cpu())


# ------------------------------------------------------------------------------------------------------- K2
def test_mpc_test_scenario(known):
    """mpc_test.py:13-56 through the drop-in classes vs the untouched reference."""
    from lq_mpc_b200.utils_class import LQ_MPC_Controller, LQ_MPC_Simulator
    A = np.array([[1, 0.7], [0.12, 0.4]]); B = np.array([[1], [1.2]])
    Q = 2 * np.eye(2); R = np.eye(1)
    x0 = np.array([0.1125, 0.19])
    F_u = np.vstack((10 * np.eye(1), -10 * np.eye(1)))
    info = LQ_MPC_Controller(20, A, B, Q, R, Q, F_u).solve(x0, np.zeros((2, 20)), np.zeros((1, 20)))
    k = known["mpc_test"]
    assert abs(info["V_N"] - k["V_N"]) < TOL * k["V_N"]
    assert info["u_0"].shape == (1,) and abs(info["u_0"][0] - k["u_0"][0]) < 1e-12
    A_true = np.array([[1.01, 0.7], [0.12, 0.41]]); B_true = np.array([[1], [1.21]])
    sim = LQ_MPC_Simulator(20, 6, A, B, Q, R, Q, F_u)
    r = sim.simulate(x0, A_true, B_true, np.zeros((2, 20)), np.zeros((1, 20)))
    assert abs(r["J_T"] - k["J_T"]) < TOL * k["J_T"]
    assert r["X"] is sim.X and r["U"] is sim.U                       # aliasing of instance buffers, as the reference
    assert np.max(np.abs(r["X"] - np.array(k["X"]))) < 1e-12
    assert np.max(np.abs(r["U"] - np.array(k["U"]))) < 1e-12


def test_random_api_cases(known):
    """Randomised reference calls (n in {2,3}, m in {1,2}): solve, simulate, energy_bound / energy_decreasing."""
    from lq_mpc_b200.control import dlqr
    from lq_mpc_b200.utils_class import LQ_MPC_Controller, LQ_MPC_Simulator, LQ_RDP_Calculator
    n_raise = 0
    for c in known["random_api"]:
        n, m, N, T = c["n"], c["m"], c["N"], c["T"]
        A, B, dA, dB = (np.array(c[k]) for k in ("A", "B", "dA", "dB"))
        Q, R = c["q"] * np.eye(n), c["r"] * np.eye(m)
        F_u = np.vstack((np.eye(m) / c["ub"], -np.eye(m) / c["ub"]))
        x0 = np.array(c["x0"])
        xr, ur = np.zeros((n, N)), np.zeros((m, N))
        sol = LQ_MPC_Controller(N, A + dA, B + dB, Q, R, Q, F_u).solve(x0, xr, ur)
        assert abs(sol["V_N"] - c["V_N"]) < TOL * abs(c["V_N"])
        assert np.max(np.abs(sol["u_0"] - np.array(c["u_0"]))) < 1e-10
        sim = LQ_MPC_Simulator(T, N, A + dA, B + dB, Q, R, Q, F_u).simulate(x0, A, B, xr, ur)
        assert abs(sim["J_T"] - c["J_T"]) < TOL * abs(c["J_T"])
        assert np.max(np.abs(sim["U"] - np.array(c["U"]))) < 1e-10
        if "K_dlqr" in c:
            K, _, _ = dlqr(A + dA, B + dB, Q, R)
            assert np.max(np.abs(K - np.array(c["K_dlqr"]))) < 1e-9 * max(1.0, np.max(np.abs(K)))
            calc = LQ_RDP_Calculator(A + dA, B + dB, Q, R, F_u)
            if "raises" in c:
                with pytest.raises(ValueError):
                    calc.energy_decreasing(N, c["e"], c["e"], -K, c["M_V"])
                n_raise += 1
            else:
                dec = calc.energy_decreasing(N, c["e"], c["e"], -K, c["M_V"])
                bnd = calc.energy_bound(N, c["e"], c["e"], x0, np.array([0.1, 1, 0.6]))
                for k, v in (("xi", dec["xi"]), ("eta", dec["eta"]), ("alpha", bnd["alpha"]), ("beta", bnd["beta"])):
                    assert abs(v - c[k]) < TOL * abs(c[k]), (k, v, c[k])
    assert n_raise > 0


def test_tracking_references(engine, tracking):
    """Non-zero x_ref / u_ref (utils_class.py:62-81): drop-in classes vs the untouched reference's answers, a batch
    through the C ABI vs the oracle's dense QP, and the state really clears (regulation answers come back)."""
    import torch
    from oracle import np_oracle as o
    from lq_mpc_b200.utils_class import LQ_MPC_Controller, LQ_MPC_Simulator
    from tests.conftest import tracking_case
    for c in map(tracking_case, tracking):
        Ah, Bh = c["A"] + c["dA"], c["B"] + c["dB"]
        sol = LQ_MPC_Controller(c["N"], Ah, Bh, c["Q"], c["R"], c["Q"], c["F_u"]).solve(c["x0"], c["x_ref"], c["u_ref"])
        assert abs(sol["V_N"] - c["V_N"]) < TOL * abs(c["V_N"]) and np.max(np.abs(sol["u_0"] - c["u_0"])) < 1e-10
        sim = LQ_MPC_Simulator(c["T"], c["N"], Ah, Bh, c["Q"], c["R"], c["Q"], c["F_u"]).simulate(
            c["x0"], c["A"], c["B"], c["x_ref"], c["u_ref"])
        assert abs(sim["J_T"] - c["J_T"]) < TOL * abs(c["J_T"])
        assert np.max(np.abs(sim["U"] - c["U"])) < 1e-10 and np.max(np.abs(sim["X"] - c["X"])) < 1e-10
    rng = np.random.default_rng(5)
    n, m, N, S = 4, 2, 6, 257
    A = rng.normal(size=(n, n)); A *= 0.9 / np.max(np.abs(np.linalg.eigvals(A)))
    B = rng.normal(size=(n, m)); Q = np.eye(n); R = 0.5 * np.eye(m)
    lo, hi = -0.55 * np.ones(m), 0.55 * np.ones(m)
    engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
    dA = rng.uniform(-0.01, 0.01, size=(n * n, S)); dB = rng.uniform(-0.01, 0.01, size=(n * m, S))
    x0 = rng.normal(size=(n, S)) * 0.5
    base = engine.mpc_solve_batch(dA, dB, N, x0=x0)
    for xr, ur in ((rng.normal(size=(n, N)) * 0.3, None), (None, rng.normal(size=(m, N)) * 0.2),
                   (rng.normal(size=(n, N + 3)) * 0.3, rng.normal(size=(m, N + 3)) * 0.2)):
        with engine.references(xr, ur):
            got = engine.mpc_solve_batch(dA, dB, N, x0=x0)
            sim = engine.simulate_batch(dA, dB, N, 5, x0=x0, want=("J_T", "U"))
        V, u0, fl = (got[k].cpu().numpy() for k in ("V", "u0", "flags"))
        J, U = sim["J_T"].cpu().numpy(), sim["U"].cpu().numpy()
        assert not np.any(fl & ~2)
        n_act = 0
        for s in range(0, S, 4):
            Ah, Bh = A + dA[:, s].reshape(n, n), B + dB[:, s].reshape(n, m)
            u_o, V_o, act = o.mpc_solve(N, Ah, Bh, Q, R, Q, lo, hi, x0[:, s], x_ref=xr, u_ref=ur)
            n_act += int(act)
            assert abs(V[0, s] - V_o) < TOL * abs(V_o) and np.max(np.abs(u0[0, :, s] - u_o)) < 1e-9
            assert bool(fl[0, s] & 2) == act
            if s % 32 == 0:
                so = o.simulate(5, N, Ah, Bh, Q, R, Q, lo, hi, x0[:, s], A, B, x_ref=xr, u_ref=ur)
                assert abs(J[s] - so["J_T"]) < TOL * abs(so["J_T"]) and np.max(np.abs(U[:, :, s].T - so["U"])) < 1e-9
        assert 0 < n_act < len(range(0, S, 4))
    with pytest.raises(Exception):
        with engine.references(np.ones((n, N - 1)), None):              # fewer than N columns
            engine.mpc_solve_batch(dA, dB, N, x0=x0)
    again = engine.mpc_solve_batch(dA, dB, N, x0=x0)                     # cleared: regulation answers, bit for bit
    assert torch.equal(again["V"], base["V"]) and torch.equal(again["u0"], base["u0"])


def test_general_input_polytope(engine, polytope):
    """F_u with rows that couple the inputs (utils_class.py:81; SURVEY 8f.3): the drop-in classes vs the untouched
    reference's answers (solve, simulate, energy_bound), a batch through the C ABI vs the dense active-set oracle, the
    bound kernel's local_radius over polytope rows vs the oracle, a box handed over as a polytope vs the box kernels,
    and the limits (rows, working-set size) failing loudly."""
    import torch
    from oracle import np_oracle as o
    from lq_mpc_b200.engine import EngineError
    from lq_mpc_b200.utils_class import LQ_MPC_Controller, LQ_MPC_Simulator, LQ_RDP_Calculator
    from tests.conftest import polytope_case, random_polytope
    n_act = 0
    for c in map(polytope_case, polytope):
        Ah, Bh = c["A"] + c["dA"], c["B"] + c["dB"]
        zx, zu = np.zeros((c["n"], c["N"])), np.zeros((c["m"], c["N"]))
        sol = LQ_MPC_Controller(c["N"], Ah, Bh, c["Q"], c["R"], c["Q"], c["F_u"]).solve(c["x0"], zx, zu)
        assert abs(sol["V_N"] - c["V_N"]) < TOL * abs(c["V_N"]) and np.max(np.abs(sol["u_0"] - c["u_0"])) < 1e-10
        sim = LQ_MPC_Simulator(c["T"], c["N"], Ah, Bh, c["Q"], c["R"], c["Q"], c["F_u"]).simulate(
            c["x0"], c["A"], c["B"], zx, zu)
        assert abs(sim["J_T"] - c["J_T"]) < TOL * abs(c["J_T"]) and np.max(np.abs(sim["U"] - c["U"])) < 1e-10
        n_act += int(np.max(c["F_u"] @ sim["U"]) > 1 - 1e-9)
        bnd = LQ_RDP_Calculator(Ah, Bh, c["Q"], c["R"], c["F_u"]).energy_bound(c["N"], c["e"], c["e"], c["x0"],
                                                                             np.array([0.1, 1, 0.6]))
        assert abs(bnd["alpha"] - c["alpha"]) < TOL * c["alpha"] and abs(bnd["beta"] - c["beta"]) < TOL * c["beta"]
    assert 4 <= n_act < len(polytope)
    rng = np.random.default_rng(9)
    for n, m, p in [(2, 2, 5), (4, 2, 8), (3, 3, 7), (4, 4, 9), (8, 2, 6)]:
        N = int(rng.integers(3, min(12, 128 // p) + 1))
        A = rng.normal(size=(n, n)); A *= 1.1 / np.max(np.abs(np.linalg.eigvals(A))); B = rng.normal(size=(n, m))
        Q, R = rng.uniform(0.5, 3) * np.eye(n), rng.uniform(0.1, 2) * np.eye(m)
        F = random_polytope(rng, m, p, 0.15, 0.45)
        engine.set_problem(A, B, Q, R, Q, None, None, 10)
        engine.set_input_polytope(F)
        S = 257
        x0 = rng.normal(size=(n, S)) * rng.uniform(0.3, 1.2)
        dA = rng.uniform(-0.02, 0.02, size=(n * n, S)); dB = rng.uniform(-0.02, 0.02, size=(n * m, S))
        got = engine.mpc_solve_batch(dA, dB, N, x0=x0)
        sim = engine.simulate_batch(dA, dB, N, 5, x0=x0, want=("J_T", "U", "flags"))
        V, u0, fl = (got[k].cpu().numpy() for k in ("V", "u0", "flags"))
        J, Us = sim["J_T"].cpu().numpy(), sim["U"].cpu().numpy()
        assert not np.any(fl & ~2) and not np.any(sim["flags"].cpu().numpy() & ~2)
        na = 0
        for s in range(0, S, 8):
            Ah, Bh = A + dA[:, s].reshape(n, n), B + dB[:, s].reshape(n, m)
            u_o, V_o, act = o.mpc_solve(N, Ah, Bh, Q, R, Q, None, None, x0[:, s], F_u=F)
            na += int(act)
            assert abs(V[0, s] - V_o) < TOL * abs(V_o) and np.max(np.abs(u0[0, :, s] - u_o)) < 1e-9
            assert bool(fl[0, s] & 2) == act
            if s % 64 == 0:
                so = o.simulate(5, N, Ah, Bh, Q, R, Q, None, None, x0[:, s], A, B, F_u=F)
                assert abs(J[s] - so["J_T"]) < TOL * abs(so["J_T"]) and np.max(np.abs(Us[:, :, s].T - so["U"])) < 1e-9
        assert na > 3
    # K3 over polytope rows (local_radius) + supplied vertex constants vs the oracle, on well-damped plants (the
    # bound formulas need rho(A + BK) + 0.4 < 1, utils.py:358)
    for n, m, p in [(2, 2, 5), (3, 2, 6), (2, 1, 2)]:
        N = 7
        A = rng.normal(size=(n, n)); A *= 0.45 / np.max(np.abs(np.linalg.eigvals(A))); B = rng.normal(size=(n, m))
        Q, R = 2.0 * np.eye(n), np.eye(m)
        F = random_polytope(rng, m, p, 0.15, 0.45) if m > 1 else np.array([[4.0], [-5.0]])
        x = rng.normal(size=n) * 0.2
        engine.set_problem(A, B, Q, R, Q, None, None, 10)
        if m > 1:
            engine.set_input_polytope(F)
        else:
            engine.set_problem(A, B, Q, R, Q, [-0.2], [0.25], 10)
        K = -o.dlqr(A, B, Q, R)[0]
        bu, bdu = o.bar_u_poly(F) if m > 1 else (o.bar_u(np.array([-0.2]), np.array([0.25])),
                                                 o.bar_d_u(np.array([-0.2]), np.array([0.25])))
        if m > 1:
            with pytest.raises(EngineError):
                engine.bounds_batch(None, None, N, 5e-3, 5e-3, 0.3, x, (0.1, 1, 0.6), 0.2, K=K, S=1)
        b = engine.bounds_batch(None, None, N, 5e-3, 5e-3, 0.3, x, (0.1, 1, 0.6), 0.2, K=K, S=1, bar_u=bu, bar_d_u=bdu)
        lo_hi = (None, None) if m > 1 else (np.array([-0.2]), np.array([0.25]))
        Fo = F if m > 1 else None
        try:
            dec = o.energy_decreasing(A, B, Q, R, *lo_hi, N, 5e-3, 5e-3, K, 0.3, F_u=Fo)
        except ValueError:                                   # math domain error in the reference's formulas
            assert int(b["flags"].cpu()[0]) & 512
            continue
        assert int(b["flags"].cpu()[0]) & ~32 == 0
        bnd = o.energy_bound(A, B, Q, R, *lo_hi, N, 5e-3, 5e-3, x, (0.1, 1, 0.6), F_u=Fo)
        for key, want in (("epsilon_K", dec["epsilon_K"]), ("xi", dec["xi"]), ("eta", dec["eta"]),
                          ("alpha", bnd["alpha"]), ("beta", bnd["beta"])):
            assert abs(float(b[key].cpu()[0]) - want) < TOL * abs(want), key
    # a box handed over as a polytope: same answers as the box kernels; clearing restores them bit for bit
    n, m, N, S = 4, 2, 6, 300
    A = rng.normal(size=(n, n)); A *= 1.1 / np.max(np.abs(np.linalg.eigvals(A))); B = rng.normal(size=(n, m))
    lo, hi = -np.array([0.2, 0.35]), np.array([0.3, 0.25])
    x0 = rng.normal(size=(n, S)); dA = rng.uniform(-.02, .02, size=(n * n, S)); dB = rng.uniform(-.02, .02, size=(n * m, S))
    engine.set_problem(A, B, np.eye(n), np.eye(m), np.eye(n), lo, hi, 10)
    box = engine.simulate_batch(dA, dB, N, 8, x0=x0, want=("J_T", "U", "flags"))
    engine.set_input_polytope(np.vstack((np.diag(1 / hi), np.diag(1 / lo))))
    pol = engine.simulate_batch(dA, dB, N, 8, x0=x0, want=("J_T", "U", "flags"))
    assert relerr(pol["J_T"].cpu().numpy(), box["J_T"].cpu().numpy()) < 1e-12
    assert torch.equal(pol["flags"], box["flags"]) and bool((box["flags"] & 2).any())
    with pytest.raises(EngineError):
        engine.set_input_polytope(np.ones((13, m)))                      # more than 12 rows
    too_long = engine.mpc_solve_batch(dA[:, :8], dB[:, :8], 70, x0=5 * x0[:, :8])   # N * p = 280 > 256
    assert bool((too_long["flags"] & 4).all()) and bool(torch.isnan(too_long["V"]).all())
    Fbox = np.vstack((np.diag(1 / hi), np.diag(1 / lo)))
    assert float((Fbox @ too_long["u0"][0].cpu().numpy()).max()) <= 1.0 + 1e-12       # shrunk onto the polytope
    engine.set_input_polytope(None)
    again = engine.simulate_batch(dA, dB, N, 8, x0=x0, want=("J_T", "U", "flags"))
    assert torch.equal(again["J_T"], box["J_T"]) and torch.equal(again["U"], box["U"])


def test_clqr_stress_vs_dense_qp(engine):
    """Heavily saturated random problems: batched K2 vs the dense Cholesky+BVLS oracle (per problem: one engine
    problem, 48 initial states)."""
    from oracle import np_oracle as o
    rng = np.random.default_rng(11)
    n_active = 0
    n_arb = 0
    for n, m in [(2, 1), (2, 2), (3, 1), (3, 2), (4, 2), (4, 1), (6, 2), (8, 2)]:
        for rep in range(3):
            N = int(rng.integers(2, min(24, 64 // m) + 1))
            A = rng.normal(size=(n, n))
            A *= rng.uniform(0.6, 1.25) / np.max(np.abs(np.linalg.eigvals(A)))
            B = rng.normal(size=(n, m))
            Mq, Mr = rng.normal(size=(n, n)), rng.normal(size=(m, m))
            Q = Mq @ Mq.T + 0.3 * np.eye(n) if rep == 2 else rng.uniform(0.5, 3) * np.eye(n)
            R = Mr @ Mr.T + 0.2 * np.eye(m) if rep == 2 else rng.uniform(0.1, 2) * np.eye(m)
            lo, hi = -rng.uniform(0.05, 0.4, size=m), rng.uniform(0.05, 0.4, size=m)
            engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
            S = 48
            x0 = rng.normal(size=(n, S)) * rng.uniform(0.2, 2.0)
            dA = rng.uniform(-0.03, 0.03, size=(n * n, S)); dB = rng.uniform(-0.03, 0.03, size=(n * m, S))
            got = engine.mpc_solve_batch(dA, dB, N, x0=x0)
            V, u0, fl = (got[k].cpu().numpy() for k in ("V", "u0", "flags"))
            assert not np.any(fl & ~2)
            n_active += int(np.sum(fl & 2) // 2)
            for s in range(0, S, 5):
                ur, Vr, _ = o.mpc_solve(N, A + dA[:, s].reshape(n, n), B + dB[:, s].reshape(n, m), Q, R, Q, lo, hi,
                                        x0[:, s], exact_fast=False)
                if abs(V[0, s] - Vr) < TOL * abs(Vr) and np.max(np.abs(u0[0, :, s] - ur)) < TOL:
                    continue
                # engine and dense-Cholesky oracle disagree beyond 1e-9: certify the oracle's active set in 50-digit
                # arithmetic and hold the ENGINE to 1e-9 against that solution
                from tests import mp_truth as mt
                Ah, Bh = A + dA[:, s].reshape(n, n), B + dB[:, s].reshape(n, m)
                H, gq, _ = o.condensed_qp(N, Ah, Bh, Q, R, Q, x0[:, s])
                z = o.box_qp(H, gq, np.tile(lo, N), np.tile(hi, N))
                ut, Vt, ok = mt.qp_truth(N, Ah, Bh, Q, R, Q, lo, hi, x0[:, s], np.flatnonzero(z <= np.tile(lo, N)),
                                         np.flatnonzero(z >= np.tile(hi, N)))
                assert ok, "oracle active set not optimal in extended precision"
                assert abs(V[0, s] - Vt) < TOL * abs(Vt) and np.max(np.abs(u0[0, :, s] - ut)) < TOL, (n, m, N, s)
                n_arb += 1
    assert n_active > 100 and n_arb <= 10


def test_clqr_long_horizon_late_saturation(engine):
    """Round 2: the cost-to-go is stored for the first 12 stages only, the stage loops load one stage ahead, ring solves
    skip the feasibility certificate. Long horizons on marginally unstable plants whose inputs saturate beyond stage 12
    (full N-stage sweep) and before it (restart from the stored S_k): batched K2 vs the dense Cholesky + BVLS oracle, and
    M_V over shared ring points == the maximum of the per-point solves."""
    from oracle import np_oracle as o
    rng = np.random.default_rng(2024)
    late = early = 0
    for (n, m) in [(2, 1), (2, 2), (3, 1), (4, 2)]:
        for rep in range(2):
            N = int(rng.integers(20, 41))
            A = rng.normal(size=(n, n))
            A *= rng.uniform(0.95, 1.15) / np.max(np.abs(np.linalg.eigvals(A)))
            B = rng.normal(size=(n, m))
            Q = rng.uniform(0.5, 3) * np.eye(n); R = rng.uniform(0.1, 2) * np.eye(m)
            lo, hi = -rng.uniform(0.02, 0.1, size=m), rng.uniform(0.02, 0.1, size=m)
            engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
            S = 40
            x0 = rng.normal(size=(n, S)) * rng.uniform(0.5, 3.0)
            got = engine.mpc_solve_batch(None, None, N, x0=x0, S=S)
            V, u0, fl = (got[k].cpu().numpy() for k in ("V", "u0", "flags"))
            assert not np.any(fl & ~2)
            for s in range(0, S, 8):
                ur, Vr, _ = o.mpc_solve(N, A, B, Q, R, Q, lo, hi, x0[:, s], exact_fast=False)
                assert abs(V[0, s] - Vr) < TOL * abs(Vr), (n, m, N, s)
                assert np.max(np.abs(u0[0, :, s] - ur)) < TOL, (n, m, N, s)
                H, gq, _ = o.condensed_qp(N, A, B, Q, R, Q, x0[:, s])
                z = o.box_qp(H, gq, np.tile(lo, N), np.tile(hi, N)).reshape(N, m)
                sat = np.flatnonzero(np.any((z <= lo + 1e-12) | (z >= hi - 1e-12), axis=1))
                if sat.size:
                    late += int(sat.max() >= 12)
                    early += int(sat.max() < 12)
            pts = x0[:, :8].T.copy()
            ring = engine.mpc_solve_batch(None, None, N, pts=pts, S=3, want=("V", "M_V"))
            Vp, MV = ring["V"].cpu().numpy(), ring["M_V"].cpu().numpy()
            assert np.max(np.abs(Vp[:, 0] - V[0, :8])) <= 1e-12 * np.max(np.abs(V[0, :8]))
            assert np.all(MV == Vp.max(axis=0))
    assert late >= 5 and early >= 1, (late, early)


def test_clqr_max_working_set_size(engine):
    """N*m = 256 is the largest working set (256-bit mask): N = 64, 128, 256 (m = 1) and N = 64, 128 with m = 2 are
    solved exactly; N*m = 257 with an active bound must flag QP_MAXITER, return V = NaN and a first input clipped into
    the box (never an approximation, never uninitialised memory), and the drop-in controller must raise on it."""
    from oracle import np_oracle as o
    from lq_mpc_b200.engine import EngineError
    from lq_mpc_b200.utils_class import LQ_MPC_Controller
    A = np.array([[1.0, 0.3], [0.0, 1.0]]); B = np.array([[0.0], [1.0]])
    engine.set_problem(A, B, np.eye(2), np.eye(1), np.eye(2), [-0.05], [0.05], 10)
    x0 = np.array([[1.0], [0.5]])
    for N in (64, 128, 256):
        got = engine.mpc_solve_batch(None, None, N, x0=x0, S=1)
        ur, Vr, act = o.mpc_solve(N, A, B, np.eye(2), np.eye(1), np.eye(2), np.array([-0.05]), np.array([0.05]),
                                  x0[:, 0], exact_fast=False)
        assert act and abs(float(got["V"][0, 0]) - Vr) < TOL * Vr and int(got["flags"][0, 0]) == 2
        assert abs(float(got["u0"][0, 0, 0]) - ur[0]) < 1e-9
    over = engine.mpc_solve_batch(None, None, 257, x0=x0, S=1)
    assert int(over["flags"][0, 0]) & 4 and math.isnan(float(over["V"][0, 0]))
    assert -0.05 <= float(over["u0"][0, 0, 0]) <= 0.05
    sim = engine.simulate_batch(None, None, 257, 3, x0=x0, S=1, want=("J_T", "U", "flags"))
    assert int(sim["flags"][0]) & 4 and float(sim["U"].abs().max()) <= 0.05
    with pytest.raises(EngineError):
        LQ_MPC_Controller(257, A, B, np.eye(2), np.eye(1), np.eye(2), np.array([[20.0], [-20.0]])).solve(
            x0[:, 0], np.zeros((2, 257)), np.zeros((1, 257)))
    B2 = np.array([[0.0, 0.1], [1.0, 0.0]])
    lo2, hi2 = np.array([-0.05, -0.2]), np.array([0.05, 0.2])
    engine.set_problem(A, B2, np.eye(2), np.eye(2), np.eye(2), lo2, hi2, 10)
    for N in (64, 128):
        got = engine.mpc_solve_batch(None, None, N, x0=x0, S=1)
        ur, Vr, act = o.mpc_solve(N, A, B2, np.eye(2), np.eye(2), np.eye(2), lo2, hi2, x0[:, 0], exact_fast=False)
        assert act and abs(float(got["V"][0, 0]) - Vr) < TOL * Vr and int(got["flags"][0, 0]) == 2


# ------------------------------------------------------------------------------------------------------- K3
def test_working_example_single(known):
    """working_example_single.py:20-108 through the drop-in modules vs the untouched reference."""
    from lq_mpc_b200 import control as ct
    from lq_mpc_b200.utils import (circle_generator, ex_stability_bounds, ex_stability_lq, fc_ec_E, fc_ec_theta,
                                   fc_omega_eta, local_radius, bar_u_solve, bar_d_u_solve)
    from lq_mpc_b200.utils_class import LQ_MPC_Controller, LQ_RDP_Behavior, LQ_RDP_Calculator
    k = known["single"]
    A = np.array([[1, 0.7], [0.12, 0.4]]); B = np.array([[1], [1.2]])
    Q = 2 * np.eye(2); R = np.eye(1); F_u = np.array([[10], [-10]])
    K_lqr, P_lqr, _ = ct.dlqr(A, B, Q, R)
    assert relerr(K_lqr, k["K_lqr"]) < TOL and relerr(P_lqr, k["P_lqr"]) < TOL
    eps = local_radius(F_u, -K_lqr, Q)
    assert abs(eps - k["epsilon_lqr"]) < TOL * eps
    x0_vec = circle_generator(8, 1.5, eps, Q)
    assert np.max(np.abs(x0_vec - np.array(k["x0_vec"]))) < 1e-12
    N = 6
    x_ref, u_ref = np.zeros((2, N)), np.zeros((1, N))
    beh = LQ_RDP_Behavior(A, B, Q, R, F_u, -K_lqr, 6, 10, -6, -2)
    M_V = beh.OL_energy_bound(N, 8, 1.5, x_ref, u_ref)
    assert abs(M_V - k["M_V"]) < TOL * M_V
    mpc = LQ_MPC_Controller(N, A, B, Q, R, Q, F_u)
    for i in range(8):
        r = mpc.solve(x0_vec[:, i], x_ref, u_ref)
        assert abs(r["V_N"] - k["ring_V"][i]) < TOL * r["V_N"]
        assert abs(r["u_0"][0] - k["ring_u0"][i][0]) < 1e-11
    ex = ex_stability_lq(A, B, Q, R, -K_lqr)
    for f in ("C_K", "lambda_K", "rho_K", "gamma", "rho_gamma"):
        assert abs(ex[f] - k["ex"][f]) < TOL * abs(k["ex"][f]), f
    bar = ex_stability_bounds(ex["gamma"], eps, M_V)
    assert bar["N_0"] == k["bar"]["N_0"] and abs(bar["L_V"] - k["bar"]["L_V"]) < TOL * bar["L_V"]
    err = fc_omega_eta(N, A, B, Q, R, -K_lqr, bar["L_V"], bar["N_0"])
    for f in ("omega_N1", "omega_N0d5", "eta", "err_th", "N_min"):
        assert abs(err[f] - k["omega_eta"][f]) < TOL * abs(k["omega_eta"][f]), f
    calc = LQ_RDP_Calculator(A, B, Q, R, F_u)
    dec = calc.energy_decreasing(N, 0.01, 0.01, -K_lqr, M_V)
    bnd = calc.energy_bound(N, 0.01, 0.01, x0_vec[:, 0], np.array([0.1, 1, 0.6]))
    assert abs(dec["xi"] - k["decrease"]["xi"]) < TOL and abs(dec["eta"] - k["decrease"]["eta"]) < TOL
    assert abs(bnd["alpha"] - k["bound"]["alpha"]) < TOL * bnd["alpha"]
    assert abs(bnd["beta"] - k["bound"]["beta"]) < TOL * bnd["beta"]
    assert bar_u_solve(F_u) == k["bar_u"] and abs(bar_d_u_solve(F_u) - k["bar_d_u"]) < 1e-15
    E = fc_ec_E(N, 0.01, 0.01, A, B, Q, R, x0_vec[:, 0], bar_u_solve(F_u), bar_d_u_solve(F_u))
    th = fc_ec_theta(N, 0.01, 0.01, A, B, 2.0)
    for f in ("E_psi", "E_u", "E_psi_u"):
        assert abs(E[f] - k["E"][f]) < TOL * abs(k["E"][f]), f
    for f in ("theta_u", "theta_x_u"):
        assert abs(th[f] - k["theta"][f]) < TOL * abs(k["theta"][f]), f


def test_extension_variant_vs_untouched_reference(extension_cases):
    """SURVEY 8f.4: LQ_RDP_Calculator.energy_decreasing_extension / utils.fc_omega_eta_extension
    (utils_class.py:375-406, utils.py:412-466) through the drop-in modules vs fourteen runs of the untouched reference
    (m = 1), including the five where the reference raises ValueError (math.log of a non-positive number)."""
    from lq_mpc_b200.utils import ex_stability_bounds, ex_stability_lq, fc_omega_eta_extension, local_radius
    from lq_mpc_b200.utils_class import LQ_RDP_Calculator
    n_raise = n_ok = 0
    for c in extension_cases:
        n = c["n"]
        A, B, K, hatK = (np.array(c[k]) for k in ("A", "B", "K", "hatK"))
        Q, R = c["q"] * np.eye(n), c["r"] * np.eye(1)
        F_u = np.array([[1 / c["ub"]], [-1 / c["ub"]]])
        calc = LQ_RDP_Calculator(A, B, Q, R, F_u)
        if "raises" in c:
            with pytest.raises(ValueError):
                calc.energy_decreasing_extension(c["N"], c["e"], c["e"], K, hatK, c["M_V"])
            n_raise += 1
            continue
        eps = local_radius(F_u, K, Q)
        bd = ex_stability_bounds(ex_stability_lq(A, B, Q, R, K)["gamma"], eps, c["M_V"])
        assert bd["N_0"] == c["N_0"] and abs(bd["L_V"] - c["L_V"]) <= TOL * c["L_V"]
        oe = fc_omega_eta_extension(c["N"], A, B, Q, R, K, hatK, bd["L_V"], bd["N_0"])
        for f in ("omega_N1", "omega_N0d5", "eta", "err_th", "N_min"):
            assert abs(oe[f] - c["omega_eta"][f]) <= TOL * abs(c["omega_eta"][f]), f
        dec = calc.energy_decreasing_extension(c["N"], c["e"], c["e"], K, hatK, c["M_V"])
        assert abs(dec["xi"] - c["xi"]) <= TOL * abs(c["xi"]) and abs(dec["eta"] - c["eta"]) <= TOL * abs(c["eta"])
        n_ok += 1
    assert n_ok >= 8 and n_raise >= 1


def test_behavior_test_scenario(known):
    """behavior_test.py:15-103 (curves + 4x4 mesh + two rings) through the drop-in LQ_RDP_Behavior."""
    from lq_mpc_b200 import control as ct
    from lq_mpc_b200.utils import circle_generator, local_radius
    from lq_mpc_b200.utils_class import LQ_RDP_Behavior
    k = known["behavior"]
    A = np.array([[1, 0.7], [0.12, 0.4]]); B = np.array([[1], [1.2]])
    Q = 2 * np.eye(2); R = np.eye(1); F_u = np.array([[10], [-10]])
    K_lqr, _, _ = ct.dlqr(A, B, Q, R)
    eps = local_radius(F_u, -K_lqr, Q)
    N = 6
    x_ref, u_ref = np.zeros((2, N)), np.zeros((1, N))
    err_nominal = {'e_A': 0.01, 'e_B': 0.01}
    p = np.array([0.1, 1, 0.6])
    beh = LQ_RDP_Behavior(A, B, Q, R, F_u, -K_lqr, 6, 10, -6, -2)
    M_V = beh.OL_energy_bound(N, 8, 1.5, x_ref, u_ref)
    x0_vec = circle_generator(8, 1.5, eps, Q)
    xi = beh.data_generation_xi(-K_lqr, M_V, N, err_nominal)
    al, be = beh.data_generation_alpha_beta(x0_vec[:, 1], p, N, err_nominal)
    for name, got in (("xi", xi), ("alpha", al), ("beta", be)):
        for part in ("error", "horizon"):
            assert relerr(got[part], k[name][part]) < TOL, (name, part)
    sys_true = {'A_true': np.array([[1.01, 0.7], [0.12, 0.41]]), 'B_true': np.array([[1], [1.21]])}
    info_ref = {'x_ref': x_ref, 'u_ref': u_ref, 'x_ref_long': np.zeros((2, 20)), 'u_ref_long': np.zeros((1, 20))}
    quad = {'x': np.array([0.12, 0.16]), 'y': np.array([0.12, 0.16])}
    mesh = beh.data_generation_mesh(N, {'T_mpc': 20, 'N_opc': 20}, sys_true, err_nominal, info_ref, M_V, p, quad)
    for f in ("X", "Y", "J_MPC_true", "J_MPC_bound", "V_OPC"):
        assert relerr(mesh[f], k["mesh"][f]) < TOL, f
    plane = beh.data_generation_plane(N, {'T_mpc': 20, 'N_opc': 20}, sys_true, err_nominal, info_ref, M_V, p, 8,
                                      np.array(k["plane_ratio"]))
    for f in ("X", "J_MPC_true", "J_MPC_bound", "V_OPC"):
        assert relerr(plane[f], k["plane"][f]) < TOL, f


def _run_data_generation(tmp_path, golden, norm_type, N_matrix, example):
    from lq_mpc_b200.utils_class import LQ_RDP_Behavior_Multiple
    np.save(tmp_path / ("error_A_%s.npy" % norm_type), golden["error_A_" + norm_type])
    np.save(tmp_path / ("error_B_%s.npy" % norm_type), golden["error_B_" + norm_type])
    old = os.getcwd()
    os.chdir(tmp_path)
    try:
        info_opc = {'A': example["A"], 'B': example["B"], 'Q': example["Q"], 'R': example["R"],
                    'F_u': np.vstack((10 * np.eye(1), -10 * np.eye(1)))}
        info_ref = {'x_ref': np.zeros([2, 7]), 'u_ref': np.zeros([1, 7]), 'x_ref_long': np.zeros([2, 30]),
                    'u_ref_long': np.zeros([1, 30])}
        beh = LQ_RDP_Behavior_Multiple(info_opc, example["info_N"], example["info_e"], N_matrix, norm_type)
        out = beh.data_generation(8, 1.5, info_ref, example["p"])
        saved = dict(np.load(tmp_path / "data_lq_mpc_multipleSys.npz"))
    finally:
        os.chdir(old)
    return out, saved


GOLDEN_KEYS = ["error", "horizon", "V_expert", "alpha_table_error", "beta_table_error", "xi_table_error",
               "bound_table_error", "true_cost_error", "alpha_table_horizon", "beta_table_horizon",
               "xi_table_horizon", "bound_table_horizon", "true_cost_horizon"]


def test_golden_file_reproduced(tmp_path, golden, example):
    """THE parity test: LQ_RDP_Behavior_Multiple.data_generation (working_example_multiple.py:98-101) on the GPU vs
    the reference's shipped data_lq_mpc_multipleSys.npz — all 13 arrays (authors' run: cvxpy/control/Gurobi)."""
    out, saved = _run_data_generation(tmp_path, golden, "f", 20, example)
    assert sorted(out.keys()) == sorted(GOLDEN_KEYS) and sorted(saved.keys()) == sorted(GOLDEN_KEYS)
    for k in GOLDEN_KEYS:
        assert np.asarray(out[k]).shape == golden[k].shape, k
        assert relerr(out[k], golden[k]) < TOL, k
        assert relerr(saved[k], golden[k]) < TOL, k
    # tighter where the reference's own third-party tolerances allow it
    assert relerr(out["true_cost_error"], golden["true_cost_error"]) < 1e-13
    assert relerr(out["alpha_table_error"], golden["alpha_table_error"]) < 1e-13


def test_norm2_grid_subset(tmp_path, golden, golden_norm2, example):
    """`_2` grids have no shipped outputs: compare with the untouched reference run on their first 5 systems."""
    out, _ = _run_data_generation(tmp_path, golden, "2", 1, example)
    for k in GOLDEN_KEYS:
        assert relerr(out[k], golden_norm2[k]) < TOL, k


def test_bounds_detail_vs_oracle(engine):
    """Every intermediate of K3 vs the oracle, m in {1,2}, general (non-scalar) Q/R in both kron conventions."""
    from oracle import np_oracle as o
    rng = np.random.default_rng(5)
    checked = 0
    for n, m in [(2, 1), (2, 2), (3, 1), (3, 2), (4, 2), (4, 1), (1, 1), (6, 2), (8, 2)]:
        for general in (False, True):
            for strict in ((True, False) if general else (True,)):
                N = int(rng.integers(1, 13))
                A = rng.normal(size=(n, n)); A *= rng.uniform(0.3, 0.9) / np.max(np.abs(np.linalg.eigvals(A)))
                B = rng.normal(size=(n, m))
                if general:
                    Mq, Mr = rng.normal(size=(n, n)), rng.normal(size=(m, m))
                    Q, R = Mq @ Mq.T + np.eye(n), Mr @ Mr.T + np.eye(m)
                else:
                    Q, R = rng.uniform(0.5, 3) * np.eye(n), rng.uniform(0.5, 2) * np.eye(m)
                lo, hi = -rng.uniform(0.05, 0.4, size=m), rng.uniform(0.05, 0.4, size=m)
                engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
                S = 6
                dA = rng.uniform(-0.01, 0.01, size=(n * n, S)); dB = rng.uniform(-0.01, 0.01, size=(n * m, S))
                e = rng.uniform(1e-4, 1e-2, size=S); MV = rng.uniform(0.05, 2.0, size=S)
                x = rng.normal(size=(n, S)) * 0.3
                p = np.array([0.1, 1, 0.6])
                got = engine.bounds_batch(dA, dB, N, e, e, MV, x, p, 0.37, strict_reference=strict, want_K=True)
                g = {k: v.cpu().numpy() for k, v in got.items()}
                for s in range(S):
                    Ah, Bh = A + dA[:, s].reshape(n, n), B + dB[:, s].reshape(n, m)
                    K, P = o.dlqr(Ah, Bh, Q, R)
                    assert np.max(np.abs(g["K"][:, s].reshape(m, n) + K)) < 1e-9 * max(1, np.max(np.abs(K)))
                    bnd = o.energy_bound(Ah, Bh, Q, R, lo, hi, N, e[s], e[s], x[:, s], p, strict_reference=strict)
                    for f, fo in (("alpha", "alpha"), ("beta", "beta"), ("E_psi", "E_psi"), ("E_u", "E_u"),
                                  ("E_psi_u", "E_psi_u"), ("min_H", "min_H"), ("norm_Gamma", "norm_Gamma"),
                                  ("theta_u", "theta_u"), ("theta_x_u", "theta_x_u")):
                        assert abs(g[f][s] - bnd[fo]) <= TOL * abs(bnd[fo]), (n, m, general, strict, f)
                    try:
                        dec = o.energy_decreasing(Ah, Bh, Q, R, lo, hi, N, e[s], e[s], -K, MV[s])
                    except ValueError:
                        assert g["flags"][s] & 512
                        continue
                    for f in ("xi", "eta", "C_K", "rho_K", "gamma", "rho_gamma", "L_V", "N_0", "omega_N1",
                              "omega_N0d5", "err_th", "N_min", "h", "epsilon_K"):
                        assert abs(g[f][s] - dec[f]) <= TOL * abs(dec[f]), (n, m, general, f)
                    den = 1 - dec["xi"] - dec["eta"]
                    bound = (bnd["alpha"] * 0.37 + bnd["beta"]) / den
                    # alpha, beta, xi, eta each hold 1e-9 (asserted above); the quotient propagates the errors of
                    # xi and eta with the computed factor (|xi| + |eta|) / |1 - xi - eta|
                    kappa = 1.0 + (abs(dec["xi"]) + abs(dec["eta"])) / abs(den)
                    assert abs(g["bound"][s] - bound) <= TOL * kappa * abs(bound)
                    checked += 1
    assert checked > 40


def test_bounds_unit_norm_branch_of_geo_M(engine):
    """geo_M's exact-equality branch `norm == 1` (utils.py:404-405) on the device: ||diag(1, 0.3)||_2 is exactly 1.0
    (geometric sum = N - 1), the neighbour 1 - 2^-30 takes the quotient branch; both vs the oracle."""
    from oracle import np_oracle as o
    for a11 in (1.0, 1.0 - 2.0 ** -30):
        A = np.diag([a11, 0.3]); B = np.array([[1.0], [0.5]]); Q = 2 * np.eye(2); R = np.eye(1)
        lo, hi = np.array([-0.1]), np.array([0.1])
        engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
        K = -o.dlqr(A, B, Q, R)[0]
        b = engine.bounds_batch(None, None, 7, 5e-3, 5e-3, 0.05, np.array([0.05, 0.02]), (0.1, 1, 0.6), 0.2, K=K, S=1)
        assert (float(b["norm_A"].cpu()[0]) == 1.0) == (a11 == 1.0)
        dec = o.energy_decreasing(A, B, Q, R, lo, hi, 7, 5e-3, 5e-3, K, 0.05)
        for key in ("xi", "eta", "omega_N1", "omega_N0d5"):
            assert abs(float(b[key].cpu()[0]) - dec[key]) <= TOL * abs(dec[key]), (a11, key)


def test_bounds_long_horizon(engine, example):
    """N = 50 (cfg-sweep upper end): 50 x 50 Gram matrix through the in-kernel tridiagonal/bisection path."""
    from oracle import np_oracle as o
    A, B, Q, R, lo, hi = (example[k] for k in ("A", "B", "Q", "R", "lo", "hi"))
    engine.set_problem(A, B, Q, R, Q, lo, hi, 30)
    rng = np.random.default_rng(2)
    S = 5
    dA = rng.uniform(-0.005, 0.005, size=(4, S)); dB = rng.uniform(-0.005, 0.005, size=(2, S))
    x = np.array([0.15, 0.1]); p = example["p"]
    for N, e in ((50, 1e-7), (23, 1e-6), (50, 5e-3)):
        got = engine.bounds_batch(dA, dB, N, e, e, 0.2, x, p, 0.2)
        g = {k: v.cpu().numpy() for k, v in got.items()}
        for s in range(S):
            Ah, Bh = A + dA[:, s].reshape(2, 2), B + dB[:, s].reshape(2, 1)
            bnd = o.energy_bound(Ah, Bh, Q, R, lo, hi, N, e, e, x, p)
            for f in ("alpha", "beta", "min_H", "norm_Gamma", "E_u"):
                assert abs(g[f][s] - bnd[f]) <= TOL * abs(bnd[f]), (N, e, f)


def test_k3_matrix_free_spectrum_matches_dense_path_and_svd(engine, monkeypatch):
    """||Gamma||_2 and lambda_min(H^) come from the matrix-free bisection of csrc/gramspec.cuh (N-stage elimination,
    no Gram matrix). It must agree with the dense route (Gram matrix + Householder + Sturm, LQMPC_K3_DENSE=1), with
    numpy's SVD of the assembled Gamma, and — general NON-scalar weights, time-major convention — with numpy's
    eigenvalues of the assembled H^ (utils.py:316-322)."""
    from oracle import np_batched as nb, np_oracle as o
    for n, m, N in [(4, 2, 10), (4, 2, 16), (2, 1, 50), (3, 3, 11), (2, 2, 33), (1, 1, 1), (2, 1, 1), (6, 2, 8)]:
        A, B, Q, R = nb.synth_problem(n, m, seed=5)
        Q, R = 1.5 * Q, 0.7 * R
        engine.set_problem(A, B, Q, R, Q, -0.3 * np.ones(m), 0.3 * np.ones(m), 10)
        dA, dB, x0 = nb.synth_samples(n, m, 67, seed=2, e=0.02)
        sA, sB, sx = _soa(dA, dB, x0)
        args = (sA, sB, N, 0.01, 0.01, 1.0, sx, (0.1, 1, 0.6), 1.0)
        new = engine.bounds_batch(*args)
        monkeypatch.setenv("LQMPC_K3_DENSE", "1")
        old = engine.bounds_batch(*args)
        monkeypatch.delenv("LQMPC_K3_DENSE")
        for k in ("norm_Gamma", "min_H", "alpha", "beta", "theta_u", "E_u"):
            assert relerr(new[k].cpu().numpy(), old[k].cpu().numpy()) < 1e-11, (n, m, N, k)
        assert np.array_equal(new["flags"].cpu().numpy(), old["flags"].cpu().numpy())
        for s in (0, 33, 66):
            G = o.sl_syn_Gamma(N, A + dA[s], B + dB[s])
            sv = np.linalg.svd(G, compute_uv=False)
            assert abs(float(new["norm_Gamma"][s]) - sv[0]) < 1e-12 * sv[0]
            assert abs(float(new["min_H"][s]) - (R[0, 0] + Q[0, 0] * sv[-1] ** 2)) < 1e-11 * R[0, 0]
    rng = np.random.default_rng(8)
    for n, m, N in [(2, 1, 40), (3, 2, 12), (4, 2, 9), (4, 4, 5)]:
        A, B, _, _ = nb.synth_problem(n, m, seed=6)
        Mq, Mr = rng.normal(size=(n, n)), rng.normal(size=(m, m))
        Q, R = Mq @ Mq.T + 0.5 * np.eye(n), Mr @ Mr.T + 0.5 * np.eye(m)
        engine.set_problem(A, B, Q, R, Q, -0.3 * np.ones(m), 0.3 * np.ones(m), 10)
        dA, dB, x0 = nb.synth_samples(n, m, 9, seed=3, e=0.02)
        got = engine.bounds_batch(*_soa(dA, dB, x0)[:2], N, 0.01, 0.01, 1.0, _soa(dA, dB, x0)[2], (0.1, 1, 0.6), 1.0,
                                  strict_reference=False)
        for s in range(9):
            H = o.hat_H(N, A + dA[s], B + dB[s], Q, R, strict_reference=False)
            ev = np.linalg.eigvalsh(0.5 * (H + H.T))
            assert abs(float(got["min_H"][s]) - ev[0]) < 1e-11 * max(ev[0], 1e-3 * ev[-1]), (n, m, N, s)


# ------------------------------------------------------------------------------------------------------- K5
@pytest.mark.parametrize("which", ["one_pass", "two_pass"])
def test_column_stats_match_numpy(engine, which):
    from lq_mpc_b200 import stats
    column_stats = stats.column_stats if which == "one_pass" else stats.column_stats_two_pass
    rng = np.random.default_rng(0)
    for cols, S in ((1, 1), (3, 7), (10, 100), (5, 100_003), (50, 20_000), (2, 3_000_001)):
        t = rng.normal(loc=0.2, scale=1e-3, size=(cols, S))
        st = column_stats(engine, t)
        assert np.array_equal(st["max"], t.max(axis=1)) and np.array_equal(st["min"], t.min(axis=1))
        assert relerr(st["mean"], t.mean(axis=1)) < 1e-12
        assert relerr(st["std"], t.std(axis=1) if S > 1 else np.zeros(cols) + 1e-300) < 1e-9 or S == 1
        assert np.all(st["count"] == S) and np.all(st["n_nonfinite"] == 0)
    t = rng.normal(size=(2, 1000)); t[0, 5] = np.inf; t[1, 7] = np.nan; t[1, 9] = -np.inf
    st = column_stats(engine, t)
    assert list(st["n_nonfinite"]) == [1, 2] and list(st["count"]) == [999, 998]
    fin = np.where(np.isfinite(t), t, np.nan)
    assert relerr(st["mean"], np.nanmean(fin, axis=1)) < 1e-12 and relerr(st["max"], np.nanmax(fin, axis=1)) == 0
    assert relerr(st["std"], np.nanstd(fin, axis=1)) < 1e-12
    # a column whose first entry is non-finite (shift falls back to 0) and a large offset (cancellation guard)
    t = 1e6 + rng.normal(scale=1e-2, size=(2, 50_001)); t[1, 0] = np.inf
    st = column_stats(engine, t)
    fin = np.where(np.isfinite(t), t, np.nan)
    assert relerr(st["mean"], np.nanmean(fin, axis=1)) < 1e-13
    assert relerr(st["std"][:1], np.nanstd(fin, axis=1)[:1]) < 1e-9     # shift = first entry: full accuracy
    empty = column_stats(engine, np.zeros((2, 0)))
    assert np.all(empty["count"] == 0) and np.all(np.isnan(empty["mean"]))


def test_k1_table_view_is_what_k5_reduces(engine):
    """eval_batch's outputs are rows of ONE contiguous table, reduced without a copy; both stats paths agree."""
    from lq_mpc_b200 import stats
    from oracle import np_batched as nb
    A, B, Q, R = nb.synth_problem(4, 2, seed=0)
    engine.set_problem(A, B, Q, R, Q, None, None, 30)
    dA, dB, x0 = nb.synth_samples(4, 2, 30_001, seed=1)
    r = engine.eval_batch(*_soa(dA, dB, x0), 9, 10)
    assert r["table"].shape == (6, 30_001) and r["table_rows"][:3] == [("J", 9), ("J", 10), ("rho", 9)]
    assert r["J"].data_ptr() == r["table"].data_ptr() and r["ratio"].data_ptr() == r["table"][4].data_ptr()
    a, b = stats.column_stats(engine, r["table"]), stats.column_stats_two_pass(engine, r["table"])
    tab = r["table"].cpu().numpy()
    for k in ("max", "min"):
        assert np.array_equal(a[k], b[k]) and np.array_equal(a[k], getattr(tab, k)(axis=1))
    assert relerr(a["mean"], tab.mean(axis=1)) < 1e-13 and relerr(b["mean"], tab.mean(axis=1)) < 1e-13
    assert relerr(a["std"], tab.std(axis=1)) < 1e-10 and relerr(b["std"], tab.std(axis=1)) < 1e-10


def test_golden_column_stats(engine, golden):
    """The reduction spec itself (utils.py:895-898) on the shipped tables."""
    from lq_mpc_b200.utils import column_statistics
    for k in ("bound_table_error", "true_cost_horizon", "xi_table_error"):
        mx, mn, mean, std = column_statistics(golden[k])
        assert np.array_equal(mx, golden[k].max(axis=0)) and np.array_equal(mn, golden[k].min(axis=0))
        assert relerr(mean, golden[k].mean(axis=0)) < 1e-13 and relerr(std, golden[k].std(axis=0)) < 1e-9


# ------------------------------------------------------------------------------------------------------- K4
@pytest.mark.parametrize("n,m,e", [(32, 8, 1e-3), (16, 4, 5e-3), (32, 8, 0.2)])
def test_k4_tiled_matches_oracle(engine, n, m, e):
    """Large-n path (CTA per sample, TMA-staged operands, warp-synchronous QR) vs the batched oracle: nested
    horizons, the single-horizon buffer plan, both compiled (n, m), and (e = 0.2) a batch with unstable closed
    loops."""
    from oracle import np_batched as nb
    A, B, Q, R = nb.synth_problem(n, m, seed=0)
    N = 30 if n == 32 else 12
    engine.set_problem_tiled(A, B, Q, R, Q, 30)
    Pexp = nb.expert_matrix(A, B, Q, R, Q, 30)
    assert relerr(engine.prepared_tiled()["Pexp"], Pexp) < 1e-11
    S = 301                                              # ragged vs the persistent grid
    dA, dB, x0 = nb.synth_samples(n, m, S, seed=1, e=e)
    ref = nb.eval_batch(A, B, Q, R, Q, Pexp, dA, dB, x0, N - 2, N)
    got = engine.eval_batch_tiled(dA, dB, x0, N - 2, N, want=("J", "rho", "ratio", "flags", "V_N"))
    g = {k: v.cpu().numpy() for k, v in got.items() if hasattr(v, "cpu")}
    assert np.array_equal((g["flags"] & 1) != 0, ref["unstable"])
    if e >= 0.2:
        assert ref["unstable"].any() and not ref["unstable"].all()
    if e < 0.2:
        assert relerr(g["rho"], ref["rho"]) < TOL and relerr(g["V_N"], ref["Vn"]) < TOL
        for k in ("J", "ratio"):
            assert relerr(g[k], ref[k]) < TOL, k
    else:
        # e = 0.2 drives the 30-step recursion of a 32-state, open-loop-unstable model to costs ~1e2-1e3; engine and
        # float64 oracle use different summation orders. Entries beyond 1e-9 are arbitrated in extended precision
        # (numpy longdouble, 64-bit mantissa: tests/mp_truth.k1_truth_ld) together with the MEASURED conditioning of the
        # sample (relative change of the value under a 1e-13 relative perturbation of dA): the engine must be within
        # max(1e-9, 64 u kappa) of the extended-precision value, and closer to it than 1e-7 in any case.
        from tests import mp_truth as mt
        for k, kr in (("V_N", "Vn"), ("J", "J"), ("rho", "rho")):
            fin = np.isfinite(ref[kr])
            err = np.where(fin, np.abs(g[k] - ref[kr]) / np.where(fin, np.abs(ref[kr]), 1.0), 0.0)
            bad = np.argwhere(err > TOL)
            worst = sorted(bad.tolist(), key=lambda hs: -err[hs[0], hs[1]])[:3]
            for h, s in worst:
                t = mt.k1_truth_ld(A, B, Q, R, Q, dA[s], dB[s], x0[s], N - 2 + h)
                key = {"V_N": "Vn", "J": "J", "rho": "rho"}[k]
                tol_s = max(TOL, 64 * 2.0 ** -53 * t["kappa_" + key])
                assert abs(g[k][h, s] - t[key]) <= min(tol_s, 1e-7) * abs(t[key]), (k, h, s, t["kappa_" + key])
            assert err.max() < 1e-6, k
    assert not np.any(g["flags"] & ~1)
    one = engine.eval_batch_tiled(dA, dB, x0, N, N)      # 3-buffer plan (A^ and P storage reused by the doubling)
    assert relerr(one["J"].cpu().numpy()[0], g["J"][2]) < 1e-12
    assert relerr(one["rho"].cpu().numpy()[0], g["rho"][2]) < 1e-12
    assert np.array_equal(one["flags"].cpu().numpy()[0], g["flags"][2])
    empty = engine.eval_batch_tiled(np.zeros((0, n, n)), np.zeros((0, n, m)), np.zeros((0, n)), N, N)
    assert empty["J"].shape == (1, 0)
    # host-buffer pipeline (3 streams, 2 slots), ragged chunks, nested horizons: identical to the device-resident call
    import torch
    h = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in (dA, dB, x0)]
    hp = engine.eval_batch_tiled_host(h[0], h[1], h[2], N - 2, N, chunk=64)
    for k in ("J", "rho", "ratio", "flags"):
        assert np.array_equal(hp[k].numpy(), g[k]), k


def test_k4_full_size_properties(engine):
    """BASELINE cfg 5 size (n = 32, m = 8, N = 30, 125 000 samples per GPU): size-independent properties instead of an
    oracle run — J is quadratic in x0 (J(2 x0) = 4 J(x0) exactly in binary FP), rho and the ratio do not depend on
    the scaling, the result does not depend on where a sample sits in the batch (persistent grid, 5 CTAs/SM), no entry
    is left pending for the QR kernel's flags, a subsample matches the oracle."""
    import torch
    from oracle import np_batched as nb
    n, m, N, S = 32, 8, 30, 125_000
    A, B, Q, R = nb.synth_problem(n, m, seed=0)
    engine.set_problem_tiled(A, B, Q, R, Q, 30)
    g = torch.Generator(device="cuda").manual_seed(11)
    dA = (torch.rand((S, n, n), device="cuda", dtype=torch.float64, generator=g) - 0.5) * 2e-3
    dB = (torch.rand((S, n, m), device="cuda", dtype=torch.float64, generator=g) - 0.5) * 2e-3
    x0 = torch.randn((S, n), device="cuda", dtype=torch.float64, generator=g)
    r1 = engine.eval_batch_tiled(dA, dB, x0, N, N)
    r2 = engine.eval_batch_tiled(dA, dB, 2.0 * x0, N, N)
    assert torch.equal(r2["J"], 4.0 * r1["J"]) and torch.equal(r2["rho"], r1["rho"])
    assert torch.equal(r2["ratio"], r1["ratio"])
    assert int((r1["flags"] != 0).sum()) == 0
    assert float(r1["ratio"].min()) >= 1.0 - 1e-9 and float(r1["rho"].max()) < 1.0
    perm = torch.randperm(S, device="cuda", generator=g)
    r3 = engine.eval_batch_tiled(dA[perm], dB[perm], x0[perm], N, N)
    assert torch.equal(r3["J"], r1["J"][:, perm]) and torch.equal(r3["rho"], r1["rho"][:, perm])
    idx = torch.arange(0, S, 997, device="cuda")
    Pexp = nb.expert_matrix(A, B, Q, R, Q, 30)
    ref = nb.eval_batch(A, B, Q, R, Q, Pexp, dA[idx].cpu().numpy(), dB[idx].cpu().numpy(), x0[idx].cpu().numpy(), N, N)
    assert relerr(r1["J"][:, idx].cpu().numpy(), ref["J"]) < TOL
    assert relerr(r1["rho"][:, idx].cpu().numpy(), ref["rho"]) < TOL
    assert relerr(r1["ratio"][:, idx].cpu().numpy(), ref["ratio"]) < TOL


def test_k4_spectral_radius_by_squaring_and_qr_fallback(engine, monkeypatch):
    """k4a's spectral radius (rescaled repeated squaring, accepted when two depths agree) vs the QR kernel on the same
    batch, and the cases squaring must NOT decide alone: a 16 x 16 Jordan block (estimates at the two depths disagree
    -> handed to the QR kernel, which is exact on a triangular matrix) and a nilpotent plant (rho = 0 exactly).
    B = 0 makes the closed loop equal to the plant, so A_cl is under the test's control."""
    from oracle import np_batched as nb
    n, m, N = 32, 8, 6
    rng = np.random.default_rng(3)
    S = 37
    x0 = rng.normal(size=(S, n))
    zA, zB = np.zeros((S, n, n)), np.zeros((S, n, m))
    for kind in ("jordan", "nilpotent"):
        sup = np.zeros(n - 1)
        sup[:15] = 0.3
        A = (0.7 * np.eye(n) + np.diag(sup, 1)) if kind == "jordan" else np.diag(0.5 * np.ones(n - 1), 1)
        B, Q, R = np.zeros((n, m)), np.eye(n), np.eye(m)
        engine.set_problem_tiled(A, B, Q, R, Q, 30)
        Pexp = nb.expert_matrix(A, B, Q, R, Q, 30)
        ref = nb.eval_batch(A, B, Q, R, Q, Pexp, zA, zB, x0, N, N)
        got = engine.eval_batch_tiled(zA, zB, x0, N, N)
        rho = got["rho"].cpu().numpy()[0]
        want = 0.7 if kind == "jordan" else 0.0
        assert np.max(np.abs(rho - want)) < 1e-13, kind
        assert relerr(got["J"].cpu().numpy(), ref["J"]) < TOL and not np.any(got["flags"].cpu().numpy())
    A, B, Q, R = nb.synth_problem(n, m, seed=0)
    engine.set_problem_tiled(A, B, Q, R, Q, 30)
    dA, dB, x0 = nb.synth_samples(n, m, 600, seed=4, e=0.05)
    monkeypatch.setenv("LQMPC_K4_RHO", "qr")
    qr = engine.eval_batch_tiled(dA, dB, x0, 30, 30)
    monkeypatch.setenv("LQMPC_K4_RHO", "sq")
    sq = engine.eval_batch_tiled(dA, dB, x0, 30, 30)
    assert relerr(sq["rho"].cpu().numpy(), qr["rho"].cpu().numpy()) < 1e-10
    assert np.array_equal(sq["flags"].cpu().numpy(), qr["flags"].cpu().numpy())
    assert np.array_equal(sq["J"].cpu().numpy(), qr["J"].cpu().numpy())
    # default: the dominant-subspace early exit (three Krylov vectors of the true closed loop, residual <= 1e-13) in
    # front of the two-estimate test — same answers, and on spectra it must NOT decide (a +- pair of equal modulus
    # next to a complex pair of the same modulus: rank 4) the later stages still deliver
    monkeypatch.delenv("LQMPC_K4_RHO")
    sub = engine.eval_batch_tiled(dA, dB, x0, 30, 30)
    assert relerr(sub["rho"].cpu().numpy(), qr["rho"].cpu().numpy()) < 1e-10
    assert np.array_equal(sub["flags"].cpu().numpy(), qr["flags"].cpu().numpy())
    assert np.array_equal(sub["J"].cpu().numpy(), qr["J"].cpu().numpy())
    dA2, dB2, x2 = nb.synth_samples(n, m, 600, seed=9, e=0.2)           # far perturbations: unstable loops included
    monkeypatch.setenv("LQMPC_K4_RHO", "qr")
    qr2 = engine.eval_batch_tiled(dA2, dB2, x2, 30, 30)
    monkeypatch.delenv("LQMPC_K4_RHO")
    sub2 = engine.eval_batch_tiled(dA2, dB2, x2, 30, 30)
    assert relerr(sub2["rho"].cpu().numpy(), qr2["rho"].cpu().numpy()) < 1e-10
    assert np.array_equal(sub2["flags"].cpu().numpy(), qr2["flags"].cpu().numpy())
    blocks = [np.array([[0.0, 0.8], [-0.8, 0.0]]), np.diag([0.8, -0.8])] + [np.array([[0.3]])] * (n - 4)
    import scipy.linalg as sla
    Tm = rng.normal(size=(n, n)) + 3 * np.eye(n)
    A4 = Tm @ sla.block_diag(*blocks) @ np.linalg.inv(Tm)
    engine.set_problem_tiled(A4, np.zeros((n, m)), np.eye(n), np.eye(m), np.eye(n), 30)
    r4 = engine.eval_batch_tiled(np.zeros((5, n, n)), np.zeros((5, n, m)), rng.normal(size=(5, n)), 6, 6)
    assert np.max(np.abs(r4["rho"].cpu().numpy() - 0.8)) < 1e-10 and not np.any(r4["flags"].cpu().numpy())


# --------------------------------------------------------------------------------------------- sweep driver (cfg 2)
def test_error_horizon_sweep_vs_golden_and_oracle(engine, golden, example):
    """Full error-level x horizon grid (lq_mpc_b200/sweep.py): column N=7 is the shipped error table, row level 4
    (e = 5e-3 = e_nominal) over N=6..10 is the shipped horizon table; N=1 and N=50 cells vs the per-sample oracle."""
    from lq_mpc_b200.sweep import QUANTITIES, error_horizon_sweep
    from oracle import np_oracle as o
    A, B, Q, R, F_u, lo, hi = (example[x] for x in ("A", "B", "Q", "R", "F_u", "lo", "hi"))
    engine.set_problem(A, B, Q, R, Q, lo, hi, 30)
    horizons = [1, 6, 7, 8, 9, 10, 50]
    eA, eB = golden["error_A_f"], golden["error_B_f"]
    r = error_horizon_sweep(engine, eA, eB, golden["error"], horizons, F_u, Q, 8, 1.5, example["p"], 30,
                            keep_tables=True)
    assert abs(r["V_expert"] - float(golden["V_expert"])) < TOL * r["V_expert"]
    assert r["evals"] == 100 * 10 * 7 and r["tables"].shape == (7, len(QUANTITIES), 10, 100)
    qi = {q: i for i, q in enumerate(QUANTITIES)}
    for q, gk in (("true_cost", "true_cost"), ("bound", "bound_table"), ("alpha", "alpha_table"),
                  ("beta", "beta_table"), ("xi", "xi_table")):
        ge = golden[gk + "_error"]; gh = golden[gk + "_horizon"]
        assert relerr(r["tables"][2, qi[q]].T, ge) < TOL, q                      # N = 7: [level][sys] -> (100, 10)
        assert relerr(r["tables"][1:6, qi[q], 4, :].T, gh) < TOL, q              # level 4, N = 6..10 -> (100, 5)
        for s, f in (("max", np.max), ("min", np.min), ("mean", np.mean), ("std", np.std)):
            assert relerr(r[q + "_" + s][:, 2], f(ge, axis=0)) < 1e-9, (q, s)    # K5 == the plotters' statistics
    assert np.allclose(r["ratio_true_max"][:, 2], golden["true_cost_error"].max(axis=0) / r["V_expert"], rtol=1e-12)
    # cells no shipped table covers: N = 1 and N = 50, three systems, two levels, vs the per-sample oracle
    x0_vec = o.circle_generator(8, 1.5, r["epsilon_lqr"], Q)
    for h, N in ((0, 1), (6, 50)):
        for i in (0, 9):
            for j in (0, 41, 99):
                try:
                    ref = o.eval_one(A + eA[:, :, j, i], B + eB[:, :, j, i], A, B, Q, R, lo, hi, N, 30,
                                     float(golden["error"][i]), x0_vec, x0_vec[:, 1], r["V_expert"], example["p"])
                except ValueError:                      # math domain error in the reference (utils.py:506-507)
                    assert r["n_invalid"][i, h] > 0
                    continue
                for q, k in (("true_cost", "J"), ("M_V", "M_V"), ("alpha", "alpha"), ("beta", "beta"), ("xi", "xi"),
                             ("eta", "eta"), ("bound", "bound")):
                    got = r["tables"][h, qi[q], i, j]
                    assert abs(got - ref[k]) <= TOL * abs(ref[k]), (N, i, j, q, got, ref[k])
    # sharded == unsharded (two shards merged by hand through the same Chan rule)
    from lq_mpc_b200 import stats as st
    parts = [error_horizon_sweep(engine, eA, eB, golden["error"], [7], F_u, Q, 8, 1.5, example["p"], 30,
                                 shard=(k, 2), keep_tables=True) for k in range(2)]
    both = np.concatenate([pp["tables"][0] for pp in parts], axis=2)
    assert np.array_equal(both, r["tables"][2])


def test_errors_are_loud(engine):
    from lq_mpc_b200.engine import EngineError
    from lq_mpc_b200.utils_class import LQ_MPC_Controller
    with pytest.raises(EngineError):
        engine.set_problem(np.eye(33), np.ones((33, 1)), np.eye(33), np.eye(1))     # n > 32: no route at all
    with pytest.raises(EngineError):
        engine.set_problem(np.eye(5), np.ones((5, 9)), np.eye(5), np.eye(9))        # m > 8
    engine.set_problem(np.eye(5), np.ones((5, 1)), np.eye(5), np.eye(1))            # run-time-dimension route
    with pytest.raises(EngineError):
        engine.set_input_polytope(np.array([[1.0], [-1.0], [0.5]]))                 # polytopes need a compiled pair
    with pytest.raises(EngineError):
        engine.eval_seeded(1, 0, 10, 0.01, 0.01, 3, 3)                              # so does the seeded entry point
    with pytest.raises(EngineError):
        LQ_MPC_Controller(3, np.eye(2), np.ones((2, 1)), np.eye(2), np.eye(1), np.eye(2),
                          np.array([[1.0, 1.0]])).solve(np.ones(2), None, None)     # F_u with 2 columns, B with 1
    with pytest.raises(EngineError):                                                  # reference window shorter than N
        LQ_MPC_Controller(3, np.eye(2), np.ones((2, 1)), np.eye(2), np.eye(1), np.eye(2),
                          np.array([[10.0], [-10.0]])).solve(np.ones(2), np.ones((2, 2)), np.zeros((1, 2)))


# ------------------------------------------------------------------------------- run-time-dimension route (any n, m)
DYN_DIMS = [(5, 1), (5, 2), (7, 3), (9, 2), (12, 4), (16, 4), (24, 6), (32, 8), (6, 4), (8, 4)]


@pytest.mark.parametrize("n,m", DYN_DIMS)
def test_dyn_k1_matches_oracle(engine, n, m):
    """(n, m) pairs WITHOUT a register-resident instantiation go through the warp-per-sample route (csrc/dyn.cuh,
    k_dyn.cu): LQ_MPC_Controller / LQ_RDP_Calculator take any (n, m) (utils_class.py:23-46, 293-306). K1 vs the
    batched oracle: nested horizons, gains, V_N, finite-T cost, flags; at n = 32, m = 8 also vs the tiled kernel (K4)."""
    from oracle import np_batched as nb
    assert (n, m) not in engine.supported_dims()
    A, B, Q, R = nb.synth_problem(n, m, seed=0)
    engine.set_problem(A, B, Q, R, Q, None, None, 30)
    S = 203
    e = 0.02 if n <= 16 else 2e-3
    dA, dB, x0 = nb.synth_samples(n, m, S, seed=1, e=e)
    Pexp = nb.expert_matrix(A, B, Q, R, Q, 30)
    assert relerr(engine.prepared()["Pexp"], Pexp) < 1e-11
    N1 = 9 if n <= 16 else 5
    ref = nb.eval_batch(A, B, Q, R, Q, Pexp, dA, dB, x0, N1 - 2, N1, T=12, want_K=True)
    got = engine.eval_batch(*_soa(dA, dB, x0), N1 - 2, N1, T=12, want=("J", "rho", "ratio", "flags", "V_N", "J_T", "K0"))
    g = {k: v.cpu().numpy() for k, v in got.items() if hasattr(v, "cpu")}
    assert np.array_equal((g["flags"] & 1) != 0, ref["unstable"]) and not np.any(g["flags"] & ~1)
    for k, kr in (("rho", "rho"), ("V_N", "Vn"), ("J_T", "JT"), ("J", "J"), ("ratio", "ratio")):
        assert relerr(g[k], ref[kr]) < TOL, k
    K = g["K0"].reshape(3, m, n, S).transpose(0, 3, 1, 2)
    assert np.max(np.abs(K - ref["K0"])) < 1e-10 * max(1.0, np.max(np.abs(ref["K0"])))
    if (n, m) == (32, 8):
        engine.set_problem_tiled(A, B, Q, R, Q, 30)
        t = engine.eval_batch_tiled(dA, dB, x0, N1, N1)
        assert relerr(t["J"].cpu().numpy()[0], g["J"][2]) < TOL and relerr(t["rho"].cpu().numpy()[0], g["rho"][2]) < TOL
    # host-buffer pipeline on the same route
    import torch
    h = [torch.from_numpy(a).pin_memory() for a in _soa(dA, dB, x0)]
    hp = engine.eval_batch_host(h[0], h[1], h[2], N1, N1, chunk=64)
    assert np.array_equal(hp["J"].numpy()[0], g["J"][2]) and np.array_equal(hp["flags"].numpy()[0], g["flags"][2])


@pytest.mark.parametrize("n,m", [(5, 1), (5, 2), (7, 3), (12, 4), (16, 4), (32, 8)])
def test_dyn_k2_box_qp_vs_dense_oracle(engine, n, m):
    """Exact input-box QP and closed loop on the run-time-dimension route vs the dense Cholesky + BVLS oracle; includes
    BASELINE cfg 5's shape (n = 32, m = 8) with the box active, which round 1 could not evaluate."""
    from oracle import np_oracle as o
    rng = np.random.default_rng(100 + n)
    N = 6 if n <= 16 else 4
    A = rng.normal(size=(n, n)); A *= 1.05 / np.max(np.abs(np.linalg.eigvals(A))); B = rng.normal(size=(n, m))
    Q, R = np.eye(n), 0.5 * np.eye(m)
    lo, hi = -0.3 * np.ones(m), 0.25 * np.ones(m)
    engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
    S = 40
    x0 = rng.normal(size=(n, S)) * (0.6 if n <= 16 else 1.5)
    dA = rng.uniform(-0.01, 0.01, size=(n * n, S)); dB = rng.uniform(-0.01, 0.01, size=(n * m, S))
    got = engine.mpc_solve_batch(dA, dB, N, x0=x0)
    V, u0, fl = (got[k].cpu().numpy() for k in ("V", "u0", "flags"))
    assert not np.any(fl & ~2)
    n_act = 0
    for s in range(0, S, 3):
        Ah, Bh = A + dA[:, s].reshape(n, n), B + dB[:, s].reshape(n, m)
        ur, Vr, act = o.mpc_solve(N, Ah, Bh, Q, R, Q, lo, hi, x0[:, s])
        n_act += int(act)
        assert abs(V[0, s] - Vr) < TOL * abs(Vr) and np.max(np.abs(u0[0, :, s] - ur)) < 1e-9, (n, m, s)
        assert bool(fl[0, s] & 2) == act
    assert n_act > 3
    ring = rng.normal(size=(4, n)) * 0.5
    mv = engine.mpc_solve_batch(dA, dB, N, pts=ring)
    Vp = mv["V"].cpu().numpy()
    assert np.array_equal(mv["M_V"].cpu().numpy(), Vp.max(axis=0))
    s = 1
    for p in range(4):
        Vr = o.mpc_solve(N, A + dA[:, s].reshape(n, n), B + dB[:, s].reshape(n, m), Q, R, Q, lo, hi, ring[p])[1]
        assert abs(Vp[p, s] - Vr) < TOL * abs(Vr)
    T = 6
    sim = engine.simulate_batch(dA, dB, N, T, x0=x0, want=("J_T", "X", "U", "flags", "n_active"))
    for s in range(0, S, 13):
        so = o.simulate(T, N, A + dA[:, s].reshape(n, n), B + dB[:, s].reshape(n, m), Q, R, Q, lo, hi, x0[:, s], A, B)
        assert abs(float(sim["J_T"][s]) - so["J_T"]) < TOL * so["J_T"]
        assert np.max(np.abs(sim["U"].cpu().numpy()[:, :, s].T - so["U"])) < 1e-9
        assert np.max(np.abs(sim["X"].cpu().numpy()[:, :, s].T - so["X"])) < 1e-9
        assert int(sim["n_active"][s]) == so["n_active"]
    if n == 5:                                                       # non-zero references on this route as well
        xr, ur = rng.normal(size=(n, N)) * 0.2, rng.normal(size=(m, N)) * 0.1
        with engine.references(xr, ur):
            trk = engine.mpc_solve_batch(dA, dB, N, x0=x0)
        for s in range(0, S, 7):
            u_o, V_o, _ = o.mpc_solve(N, A + dA[:, s].reshape(n, n), B + dB[:, s].reshape(n, m), Q, R, Q, lo, hi,
                                      x0[:, s], x_ref=xr, u_ref=ur)
            assert abs(float(trk["V"][0, s]) - V_o) < TOL * abs(V_o)
            assert np.max(np.abs(trk["u0"].cpu().numpy()[0, :, s] - u_o)) < 1e-9


@pytest.mark.parametrize("n,m", [(5, 1), (5, 2), (7, 3), (12, 4), (16, 4), (32, 8)])
def test_dyn_k3_bounds_and_dlqr_vs_oracle(engine, n, m):
    """dlqr (DARE by doubling), norms, matrix-free Gram spectrum and the bound formulas on the run-time-dimension route
    vs the per-sample oracle — energy_bound / energy_decreasing at n = 16 and n = 32 (BASELINE cfg 5's shape)."""
    from oracle import np_oracle as o
    rng = np.random.default_rng(200 + n)
    N = 7 if n <= 16 else 5
    A = rng.normal(size=(n, n)); A *= 0.5 / np.max(np.abs(np.linalg.eigvals(A))); B = rng.normal(size=(n, m))
    Q, R = 2.0 * np.eye(n), np.eye(m)
    lo, hi = -0.2 * np.ones(m), 0.3 * np.ones(m)
    engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
    pr = engine.prepared()
    assert relerr(pr["Qinv"], np.linalg.inv(Q)) < 1e-12 and abs(pr["maxQ"] - 2.0) < 1e-12 and abs(pr["minR"] - 1.0) < 1e-12
    S = 7
    dA = rng.uniform(-0.005, 0.005, size=(n * n, S)); dB = rng.uniform(-0.005, 0.005, size=(n * m, S))
    d = engine.dlqr_batch(dA, dB)
    e = rng.uniform(1e-4, 5e-3, size=S); MV = rng.uniform(0.05, 1.0, size=S)
    x = rng.normal(size=(n, S)) * 0.2
    p = np.array([0.1, 1, 0.6])
    got = engine.bounds_batch(dA, dB, N, e, e, MV, x, p, 0.37, want_K=True, want_P=True)
    g = {k: v.cpu().numpy() for k, v in got.items()}
    for s in range(S):
        Ah, Bh = A + dA[:, s].reshape(n, n), B + dB[:, s].reshape(n, m)
        K, P = o.dlqr(Ah, Bh, Q, R)
        assert np.max(np.abs(d["K"].cpu().numpy()[:, s].reshape(m, n) - K)) < 1e-9 * max(1, np.max(np.abs(K)))
        assert np.max(np.abs(d["P"].cpu().numpy()[:, s].reshape(n, n) - P)) < 1e-9 * np.max(np.abs(P))     # normwise
        assert np.max(np.abs(g["K"][:, s].reshape(m, n) + K)) < 1e-9 * max(1, np.max(np.abs(K)))
        bnd = o.energy_bound(Ah, Bh, Q, R, lo, hi, N, e[s], e[s], x[:, s], p)
        for f in ("alpha", "beta", "E_psi", "E_u", "E_psi_u", "min_H", "norm_Gamma", "theta_u", "theta_x_u"):
            assert abs(g[f][s] - bnd[f]) <= TOL * abs(bnd[f]), (n, m, f)
        try:
            dec = o.energy_decreasing(Ah, Bh, Q, R, lo, hi, N, e[s], e[s], -K, MV[s])
        except ValueError:
            assert g["flags"][s] & 512
            continue
        for f in ("xi", "eta", "C_K", "rho_K", "gamma", "rho_gamma", "L_V", "N_0", "omega_N1", "omega_N0d5",
                  "err_th", "N_min", "h", "epsilon_K"):
            assert abs(g[f][s] - dec[f]) <= TOL * abs(dec[f]), (n, m, f)
    # general (non-scalar) weights in the time-major convention, and a supplied shared gain
    Mq, Mr = rng.normal(size=(n, n)), rng.normal(size=(m, m))
    Q2, R2 = Mq @ Mq.T / n + np.eye(n), Mr @ Mr.T / m + np.eye(m)
    engine.set_problem(A, B, Q2, R2, Q2, lo, hi, 10)
    Ksh = -o.dlqr(A, B, Q2, R2)[0]
    g2 = engine.bounds_batch(dA, dB, N, 1e-3, 1e-3, 0.3, x[:, 0], p, 0.2, K=Ksh, strict_reference=False)
    for s in range(0, S, 3):
        Ah, Bh = A + dA[:, s].reshape(n, n), B + dB[:, s].reshape(n, m)
        bnd = o.energy_bound(Ah, Bh, Q2, R2, lo, hi, N, 1e-3, 1e-3, x[:, 0], p, strict_reference=False)
        for f in ("alpha", "beta", "min_H", "norm_Gamma"):
            assert abs(float(g2[f][s]) - bnd[f]) <= TOL * abs(bnd[f]), (n, m, f)


def test_dyn_dropin_classes_with_five_states():
    """The drop-in classes on a 5-state, 2-input plant (no compiled pair): solve / simulate / energy_bound vs the oracle."""
    from oracle import np_oracle as o
    from lq_mpc_b200.control import dlqr
    from lq_mpc_b200.utils_class import LQ_MPC_Controller, LQ_MPC_Simulator, LQ_RDP_Calculator
    rng = np.random.default_rng(3)
    n, m, N, T = 5, 2, 6, 8
    A = rng.normal(size=(n, n)); A *= 0.6 / np.max(np.abs(np.linalg.eigvals(A))); B = rng.normal(size=(n, m))
    Q, R = 1.5 * np.eye(n), np.eye(m)
    ub = 0.2
    F_u = np.vstack((np.eye(m) / ub, -np.eye(m) / ub))
    lo, hi = -ub * np.ones(m), ub * np.ones(m)
    x0 = rng.normal(size=n) * 0.8
    sol = LQ_MPC_Controller(N, A, B, Q, R, Q, F_u).solve(x0, np.zeros((n, N)), np.zeros((m, N)))
    ur, Vr, act = o.mpc_solve(N, A, B, Q, R, Q, lo, hi, x0)
    assert act and abs(sol["V_N"] - Vr) < TOL * Vr and np.max(np.abs(sol["u_0"] - ur)) < 1e-9
    At = A + rng.uniform(-0.01, 0.01, size=(n, n))
    sim = LQ_MPC_Simulator(T, N, A, B, Q, R, Q, F_u).simulate(x0, At, B, np.zeros((n, N)), np.zeros((m, N)))
    so = o.simulate(T, N, A, B, Q, R, Q, lo, hi, x0, At, B)
    assert abs(sim["J_T"] - so["J_T"]) < TOL * so["J_T"] and np.max(np.abs(sim["U"] - so["U"])) < 1e-9
    K, P, _ = dlqr(A, B, Q, R)
    Ko, Po = o.dlqr(A, B, Q, R)
    assert relerr(K, Ko) < 1e-9 and relerr(P, Po) < 1e-9
    calc = LQ_RDP_Calculator(A, B, Q, R, F_u)
    bnd = calc.energy_bound(N, 5e-3, 5e-3, x0, np.array([0.1, 1, 0.6]))
    bo = o.energy_bound(A, B, Q, R, lo, hi, N, 5e-3, 5e-3, x0, (0.1, 1, 0.6))
    assert abs(bnd["alpha"] - bo["alpha"]) < TOL * bo["alpha"] and abs(bnd["beta"] - bo["beta"]) < TOL * bo["beta"]
    dec = calc.energy_decreasing(N, 5e-3, 5e-3, -K, 0.4)
    do = o.energy_decreasing(A, B, Q, R, lo, hi, N, 5e-3, 5e-3, -Ko, 0.4)
    assert abs(dec["xi"] - do["xi"]) < TOL * do["xi"] and abs(dec["eta"] - do["eta"]) < TOL * abs(do["eta"])
