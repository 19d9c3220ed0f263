"""GPU coverage of what the per-sample parity tests (tests/test_gpu_parity.py) leave open: every compiled (n, m)
instantiation of every entry point, and launches in which each thread or warp handles several samples in turn.

  A. Instantiation matrix: box solves, ring points, closed loops, references, polytopes, bounds and dlqr at each of the
     pairs of engine.supported_dims(), seeded K1 at the pairs the parity tests leave out — vs the float64 oracle.
  B. Multi-sample launches: batches of at least four samples per launched thread (per warp on the run-time-dimension
     route), deeply saturating and tiny initial states interleaved so that consecutive samples of a thread leave very
     different scratch behind. A gathered subset and a permutation of the batch must reproduce the outputs bit for bit
     (the per-sample arithmetic does not depend on where a sample sits), as must the same call after one with a larger
     horizon (the workspace is then re-reserved with another layout); a subsample, the last sample included, must
     match the oracle.
  C. The host-buffer pipeline on every K1 build, with a ragged last chunk, bit for bit against the device-resident call.

Tolerance 1e-9 relative, as in the parity tests; where the engine and the float64 oracle disagree beyond it, the solve is
arbitrated in 50-digit arithmetic (tests/mp_truth.py).
"""
import numpy as np
import pytest

from tests.conftest import random_polytope, relerr

pytestmark = pytest.mark.gpu
TOL = 1e-9
# literal list of the compiled pairs: a pair added to LQ_FOR_EACH_DIM fails test_every_compiled_pair_is_covered until
# it is added here as well
ALL_DIMS = [(1, 1), (2, 1), (2, 2), (3, 1), (3, 2), (3, 3), (4, 1), (4, 2), (4, 4), (6, 2), (8, 2)]
P3 = np.array([0.1, 1, 0.6])


def _plant(rng, n, m, general, radius=(0.6, 1.0)):
    A = rng.normal(size=(n, n)); A *= rng.uniform(*radius) / np.max(np.abs(np.linalg.eigvals(A)))
    B = rng.normal(size=(n, m))
    if general:
        Mq, Mr = rng.normal(size=(n, n)), rng.normal(size=(m, m))
        Q, R = Mq @ Mq.T / n + 0.5 * np.eye(n), Mr @ Mr.T / m + 0.3 * np.eye(m)
    else:
        Q, R = rng.uniform(0.5, 3) * np.eye(n), rng.uniform(0.1, 2) * np.eye(m)
    lo, hi = -rng.uniform(0.05, 0.4, size=m), rng.uniform(0.05, 0.4, size=m)
    return A, B, Q, R, lo, hi


def _scaled_states(A, B, Q, R, N, lo, hi, d, t):
    """Columns of d (torch, [n][S]) rescaled so that the unconstrained plan of the nominal model peaks at t[s] times the
    input box: t > 1 saturates, t < 1 stays inside (the plan is linear in the state). Runs on d's device."""
    import torch
    from oracle import np_oracle as o
    K, _ = o.riccati(A, B, Q, R, Q, N)
    T = lambda a: torch.as_tensor(a, dtype=torch.float64, device=d.device)   # noqa: E731
    At, Bt, lo_t, hi_t = T(A), T(B), T(lo)[:, None], T(hi)[:, None]
    x, r = d.clone(), torch.zeros(d.shape[1], dtype=torch.float64, device=d.device)
    for k in range(N):
        u = T(K[k]) @ x
        r = torch.maximum(r, torch.maximum(u / hi_t, u / lo_t).amax(0))
        x = At @ x + Bt @ u
    return d * (T(t) / r)


def _model(A, B, dA, dB, s):
    n, m = B.shape
    return A + dA[:, s].reshape(n, n), B + dB[:, s].reshape(n, m)


def _check_solve(N, Ah, Bh, Q, R, lo, hi, x0, V, u0, fl, x_ref=None, u_ref=None, F_u=None):
    """Engine's V, u0 and active flag (bit 2) of one solve vs the oracle; returns (active, arbitrated). A box regulation
    solve that misses 1e-9 is held to the 50-digit solution of the oracle's active set instead (as
    test_clqr_stress_vs_dense_qp does)."""
    from oracle import np_oracle as o
    kw = dict(x_ref=x_ref, u_ref=u_ref, F_u=F_u)
    ur, Vr, act = o.mpc_solve(N, Ah, Bh, Q, R, Q, lo, hi, x0, **kw)
    plain = x_ref is None and u_ref is None and F_u is None
    if plain and not act:
        ur, Vr, _ = o.mpc_solve(N, Ah, Bh, Q, R, Q, lo, hi, x0, exact_fast=False)
    assert bool(fl & 2) == act
    if abs(V - Vr) < TOL * abs(Vr) and np.max(np.abs(u0 - ur)) < TOL:
        return act, False
    assert plain, "engine and oracle disagree: V %r vs %r, u0 %r vs %r" % (V, Vr, u0, ur)
    from tests import mp_truth as mt
    H, gq, _ = o.condensed_qp(N, Ah, Bh, Q, R, Q, x0)
    z = o.box_qp(H, gq, np.tile(lo, N), np.tile(hi, N))
    ut, Vt, ok = mt.qp_truth(N, Ah, Bh, Q, R, Q, lo, hi, x0, np.flatnonzero(z <= np.tile(lo, N)),
                             np.flatnonzero(z >= np.tile(hi, N)))
    assert ok, "oracle active set not optimal in extended precision"
    assert abs(V - Vt) < TOL * abs(Vt) and np.max(np.abs(u0 - ut)) < TOL
    return act, True


def _check_sim(T, N, Ah, Bh, Q, R, lo, hi, x0, A, B, J, X, U, n_act, F_u=None):
    from oracle import np_oracle as o
    so = o.simulate(T, N, Ah, Bh, Q, R, Q, lo, hi, x0, A, B, F_u=F_u)
    assert abs(J - so["J_T"]) < TOL * so["J_T"]
    if U is not None:
        assert np.max(np.abs(U - so["U"])) < TOL
    if X is not None:
        assert np.max(np.abs(X - so["X"])) < TOL * max(1.0, np.max(np.abs(so["X"])))
    if n_act is not None:
        assert n_act == so["n_active"]
    return so["n_active"]


def _check_bounds(g, s, Ah, Bh, Q, R, lo, hi, N, e, MV, x, V_expert, strict=True):
    """Every K3 field test_bounds_detail_vs_oracle checks, for sample s of the engine's outputs g (numpy)."""
    from oracle import np_oracle as o
    n, m = Bh.shape
    K, P = o.dlqr(Ah, Bh, Q, R)
    assert np.max(np.abs(g["K"][:, s].reshape(m, n) + K)) < TOL * max(1, np.max(np.abs(K)))
    if "P" in g:
        assert np.max(np.abs(g["P"][:, s].reshape(n, n) - P)) < TOL * np.max(np.abs(P))
    bnd = o.energy_bound(Ah, Bh, Q, R, lo, hi, N, e, e, x, P3, strict_reference=strict)
    for f in ("alpha", "beta", "E_psi", "E_u", "E_psi_u", "min_H", "norm_Gamma", "theta_u", "theta_x_u"):
        assert abs(g[f][s] - bnd[f]) <= TOL * abs(bnd[f]), f
    try:
        dec = o.energy_decreasing(Ah, Bh, Q, R, lo, hi, N, e, e, -K, MV)
    except ValueError:                                 # math domain error in the reference's formulas
        assert g["flags"][s] & 512
        return False
    for f in ("xi", "eta", "C_K", "rho_K", "gamma", "rho_gamma", "L_V", "N_0", "omega_N1", "omega_N0d5", "err_th",
              "N_min", "h", "epsilon_K"):
        assert abs(g[f][s] - dec[f]) <= TOL * abs(dec[f]), f
    den = 1 - dec["xi"] - dec["eta"]
    bound = (bnd["alpha"] * V_expert + bnd["beta"]) / den
    kappa = 1.0 + (abs(dec["xi"]) + abs(dec["eta"])) / abs(den)
    assert abs(g["bound"][s] - bound) <= TOL * kappa * abs(bound)
    return True


def _same_bits(a, b):
    """Bit-for-bit equality, NaN payloads included (K3 outputs are NaN where the formulas have no value)."""
    import torch
    if a.dtype == torch.float64:
        a, b = a.view(torch.int64), b.view(torch.int64)
    return torch.equal(a, b)


def _np(d):
    return {k: v.cpu().numpy() for k, v in d.items() if hasattr(v, "cpu")}


# ===================================================================================== A. instantiation matrix
def test_every_compiled_pair_is_covered(engine):
    assert engine.supported_dims() == ALL_DIMS


@pytest.mark.parametrize("n,m", ALL_DIMS)
def test_box_solve_ring_and_closed_loop_every_pair(engine, n, m):
    """Box K2 at every compiled pair: per-sample solves at a short (whole cost-to-go stored) and a long horizon (full
    sweep and restart from the stored S_k), scalar and general SPD weights, most states saturating; M_V over ring points
    == the per-column maximum of V bit for bit; closed loops (X, U, J_T, flags, n_active) that end inside the
    certificate ellipsoid — the branch that re-reads the stage-0 gain from scratch at (3,3), (4,4), (6,2), (8,2) —
    and the shared-state call == the per-sample call with the state tiled, bit for bit."""
    import torch
    rng = np.random.default_rng(1000 + 10 * n + m)
    S, T = 64, 30
    for N, general in ((int(rng.integers(3, 12)), False), (int(rng.integers(20, min(40, 256 // m) + 1)), True)):
        A, B, Q, R, lo, hi = _plant(rng, n, m, general)
        engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
        dA = rng.uniform(-0.005, 0.005, size=(n * n, S)); dB = rng.uniform(-0.005, 0.005, size=(n * m, S))
        t = np.where(np.arange(S) % 4 == 0, rng.uniform(0.2, 0.7, S), rng.uniform(1.3, 3.0, S))
        x0 = _scaled_states(A, B, Q, R, N, lo, hi, torch.as_tensor(rng.normal(size=(n, S))), t).numpy()
        g = _np(engine.mpc_solve_batch(dA, dB, N, x0=x0))
        assert not np.any(g["flags"] & ~2)
        n_act = 0
        for s in range(0, S, 3):
            n_act += _check_solve(N, *_model(A, B, dA, dB, s), Q, R, lo, hi, x0[:, s], g["V"][0, s], g["u0"][0, :, s],
                                  g["flags"][0, s])[0]
        assert 0 < n_act < len(range(0, S, 3)), (N, n_act)
        pts = x0[:, :4].T.copy()
        ring = _np(engine.mpc_solve_batch(dA, dB, N, pts=pts))
        assert np.array_equal(ring["M_V"], ring["V"].max(axis=0))
        for s in (0, 31, S - 1):
            for p in range(4):
                _check_solve(N, *_model(A, B, dA, dB, s), Q, R, lo, hi, pts[p], ring["V"][p, s], ring["u0"][p, :, s],
                             ring["flags"][p, s])
        want = ("J_T", "X", "U", "flags", "n_active")
        sim = _np(engine.simulate_batch(dA, dB, N, T, x0=x0, want=want))
        assert not np.any(sim["flags"] & ~2)
        settled = 0
        for s in range(1, S, 9):
            na = _check_sim(T, N, *_model(A, B, dA, dB, s), Q, R, lo, hi, x0[:, s], A, B, sim["J_T"][s],
                            sim["X"][:, :, s].T, sim["U"][:, :, s].T, sim["n_active"][s])
            settled += int(0 < na < T - 5)
        assert settled >= 2, (N, settled)               # saturated first, then many steps inside the box
        sh = engine.simulate_batch(dA, dB, N, T, x0_shared=x0[:, 1], want=want)
        tl = engine.simulate_batch(dA, dB, N, T, x0=np.repeat(x0[:, 1:2], S, axis=1), want=want)
        for k in want:
            assert torch.equal(sh[k], tl[k]), k


@pytest.mark.parametrize("n,m", ALL_DIMS)
def test_references_and_polytope_every_pair(engine, n, m):
    """Non-zero references (affine law) at every compiled pair; for m >= 2 a random input polytope, solve and closed
    loop; all vs the dense oracle."""
    import torch
    rng = np.random.default_rng(2000 + 10 * n + m)
    N, S = int(rng.integers(5, 12)), 48
    A, B, Q, R, lo, hi = _plant(rng, n, m, general=bool(n % 2))
    engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
    dA = rng.uniform(-0.01, 0.01, size=(n * n, S)); dB = rng.uniform(-0.01, 0.01, size=(n * m, S))
    t = np.where(np.arange(S) % 4 == 0, 0.3, 2.0)
    x0 = _scaled_states(A, B, Q, R, N, lo, hi, torch.as_tensor(rng.normal(size=(n, S))), t).numpy()
    # references small beside the states, so that saturating and inside-the-box solves both remain
    xr = rng.normal(size=(n, N + 2)) * 0.1 * np.median(np.abs(x0[:, ::4]))
    ur = rng.normal(size=(m, N + 2)) * 0.1 * np.min(hi)
    with engine.references(xr, ur):
        g = _np(engine.mpc_solve_batch(dA, dB, N, x0=x0))
    assert not np.any(g["flags"] & ~2)
    n_act = sum(_check_solve(N, *_model(A, B, dA, dB, s), Q, R, lo, hi, x0[:, s], g["V"][0, s], g["u0"][0, :, s],
                             g["flags"][0, s], x_ref=xr, u_ref=ur)[0] for s in range(0, S, 3))
    assert 0 < n_act < len(range(0, S, 3)), n_act
    if m < 2:
        return
    p = 2 * m + 1
    F = random_polytope(rng, m, p, 0.15, 0.45)
    engine.set_problem(A, B, Q, R, Q, None, None, 10)
    engine.set_input_polytope(F)
    x0 = 2.0 * x0
    g = _np(engine.mpc_solve_batch(dA, dB, N, x0=x0))
    sim = _np(engine.simulate_batch(dA, dB, N, 6, x0=x0, want=("J_T", "U", "flags")))
    engine.set_input_polytope(None)
    assert not np.any(g["flags"] & ~2) and not np.any(sim["flags"] & ~2)
    n_act = 0
    for s in range(0, S, 3):
        Ah, Bh = _model(A, B, dA, dB, s)
        n_act += _check_solve(N, Ah, Bh, Q, R, None, None, x0[:, s], g["V"][0, s], g["u0"][0, :, s], g["flags"][0, s],
                              F_u=F)[0]
        if s % 12 == 0:
            _check_sim(6, N, Ah, Bh, Q, R, None, None, x0[:, s], A, B, sim["J_T"][s], None, sim["U"][:, :, s].T, None,
                       F_u=F)
    assert n_act > 0


@pytest.mark.parametrize("n,m", ALL_DIMS)
def test_bounds_and_dlqr_every_pair(engine, n, m):
    """K3 at every compiled pair — every detail field, the gain K_out and the DARE solution P_out vs the oracle, scalar
    and general weights in both kron conventions — and dlqr_batch on 129 samples (K to 1e-9, P normwise, flags 0)."""
    from oracle import np_oracle as o
    rng = np.random.default_rng(3000 + 10 * n + m)
    checked = 0
    for general, strict in ((False, True), (True, True), (True, False)):
        N = int(rng.integers(2, 13))
        A, B, Q, R, lo, hi = _plant(rng, n, m, general, radius=(0.2, 0.5))
        engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
        S = 6
        dA = rng.uniform(-0.01, 0.01, size=(n * n, S)); dB = rng.uniform(-0.01, 0.01, size=(n * m, S))
        e = rng.uniform(1e-4, 1e-2, size=S); MV = rng.uniform(0.05, 2.0, size=S)
        x = rng.normal(size=(n, S)) * 0.3
        g = _np(engine.bounds_batch(dA, dB, N, e, e, MV, x, P3, 0.37, strict_reference=strict, want_K=True,
                                    want_P=True))
        for s in range(S):
            checked += _check_bounds(g, s, *_model(A, B, dA, dB, s), Q, R, lo, hi, N, e[s], MV[s], x[:, s], 0.37,
                                     strict)
    assert checked >= 6             # energy_decreasing defined (no math domain error) on a third of the samples or more
    S = 129
    dA = rng.uniform(-0.01, 0.01, size=(n * n, S)); dB = rng.uniform(-0.01, 0.01, size=(n * m, S))
    d = _np(engine.dlqr_batch(dA, dB))
    assert not d["flags"].any()
    for s in range(S):
        K, P = o.dlqr(*_model(A, B, dA, dB, s), Q, R)
        assert np.max(np.abs(d["K"][:, s].reshape(m, n) - K)) < TOL * max(1, np.max(np.abs(K))), s
        assert np.max(np.abs(d["P"][:, s].reshape(n, n) - P)) < TOL * np.max(np.abs(P)), s


@pytest.mark.parametrize("n,m", [(1, 1), (2, 2), (3, 1), (3, 2), (3, 3), (4, 1), (4, 4)])
def test_eval_seeded_remaining_pairs(engine, n, m):
    """lqmpc_eval_seeded at the pairs test_gpu_parity.py does not run it on, over an index range that crosses 2^32, vs
    the oracle on the numpy restatement of the in-kernel Philox stream."""
    from oracle import np_batched as nb, np_sampler as ns
    A, B, Q, R = nb.synth_problem(n, m, seed=4)
    engine.set_problem(A, B, Q, R, Q, None, None, 30)
    S, first = 3001, (1 << 32) - 1234
    got = _np(engine.eval_seeded(5, first, S, 0.01, 0.005, 8, 10, want=("J", "rho", "ratio", "flags")))
    dA, dB, x0 = ns.seeded_samples(5, first, S, n, m, 0.01, 0.005)
    ref = nb.eval_batch(A, B, Q, R, Q, nb.expert_matrix(A, B, Q, R, Q, 30), dA, dB, x0, 8, 10)
    assert np.array_equal((got["flags"] & 1) != 0, ref["unstable"]) and not np.any(got["flags"] & ~1)
    for k in ("J", "rho", "ratio"):
        assert relerr(got[k], ref[k]) < TOL, k


# ===================================================================================== B. multi-sample launches
def _sizes():
    import torch
    pr = torch.cuda.get_device_properties(0)
    k2 = 4 * pr.multi_processor_count * pr.max_threads_per_multi_processor       # K2 at one wave, any occupancy
    k3 = 4 * pr.multi_processor_count * 8 * 128                                  # dense K3: SMs x 8 CTAs of 128
    warp = 4 * pr.multi_processor_count * pr.max_threads_per_multi_processor // 32   # one sample per warp
    return k2, k3, warp


def _layout_invariance(call, S, N, N_big, seed):
    """call(cols, N) -> dict of device tensors with the sample axis last, on the batch gathered at `cols` (a device index
    tensor; None = the whole batch in order). Returns the whole-batch outputs and ~300 indices (the last sample
    included) for the oracle."""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    full = call(None, N)
    rng = np.random.default_rng(seed)
    sub = np.unique(np.r_[np.arange(300), np.arange(S - 300, S), rng.choice(S, 1400, replace=False)])
    sub_t = torch.as_tensor(sub, device="cuda")
    part = call(sub_t, N)                                 # every sample on its own thread
    for k, v in part.items():
        assert _same_bits(v, full[k][..., sub_t]), ("subset", k)
    perm = torch.randperm(S, device="cuda", generator=g)
    pm = call(perm, N)
    for k, v in pm.items():
        assert _same_bits(v, full[k][..., perm]), ("permutation", k)
    del pm
    call(None, N_big)                                     # larger scratch, another layout
    again = call(None, N)
    for k, v in again.items():
        assert _same_bits(v, full[k]), ("after a larger horizon", k)
    del again
    return full, np.unique(np.r_[rng.choice(S - 1, 299, replace=False), S - 1])


def _batch(n, m, S, seed, e=0.005):
    """Device SoA perturbations [n*n][S], [n*m][S], random state directions [n][S] and a random half of the batch flagged
    `deep` (the other half tiny)."""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    dA = (torch.rand((n * n, S), device="cuda", dtype=torch.float64, generator=g) - 0.5) * (2 * e)
    dB = (torch.rand((n * m, S), device="cuda", dtype=torch.float64, generator=g) - 0.5) * (2 * e)
    d = torch.randn((n, S), device="cuda", dtype=torch.float64, generator=g)
    deep = torch.rand(S, device="cuda", dtype=torch.float64, generator=g) < 0.5
    return dA, dB, d, deep


def _cols(t, cols):
    return t if cols is None else t[..., cols]


K2_PAIRS = [(2, 1, 24), (4, 2, 20), (8, 2, 12)]


@pytest.mark.parametrize("n,m,N", K2_PAIRS)
def test_k2_box_multi_sample_launch(engine, n, m, N, monkeypatch):
    """Box K2 with every launched thread striding over >= 4 samples (LQMPC_K2_WAVES=1, batch >= 4 x SMs x threads per
    SM), deep (x 5 the saturation scale) and tiny states interleaved: per-sample solves, ring points (a deep and a tiny
    point in turn), closed loops from per-sample and from shared states — layout invariance and the oracle."""
    import torch
    monkeypatch.setenv("LQMPC_K2_WAVES", "1")
    S = _sizes()[0]
    rng = np.random.default_rng(4000 + n)
    A, B, Q, R, lo, hi = _plant(rng, n, m, general=(n == 4), radius=(0.85, 0.95))
    engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
    dA, dB, d, deep = _batch(n, m, S, seed=n)
    x0 = _scaled_states(A, B, Q, R, N, lo, hi, d, torch.where(deep, 5.0, 0.02))
    cpu = lambda t, idx: t[..., torch.as_tensor(idx, device="cuda")].cpu().numpy()   # noqa: E731

    def oracle_inputs(oi):
        return cpu(dA, oi), cpu(dB, oi), cpu(x0, oi)

    # per-sample solves
    full, oi = _layout_invariance(lambda c, N_: engine.mpc_solve_batch(_cols(dA, c), _cols(dB, c), N_, x0=_cols(x0, c)),
                                  S, N, N + 9, seed=1)
    g = {k: v[..., oi].cpu().numpy() for k, v in full.items()}
    dA_o, dB_o, x_o = oracle_inputs(oi)
    assert not np.any(g["flags"] & ~2)
    n_act = sum(_check_solve(N, *_model(A, B, dA_o, dB_o, i), Q, R, lo, hi, x_o[:, i], g["V"][0, i], g["u0"][0, :, i],
                             g["flags"][0, i])[0] for i in range(len(oi)))
    assert 0.3 * len(oi) < n_act < 0.7 * len(oi)
    # ring points: deep and tiny alternate inside every sample
    pts = torch.stack([x0[:, deep][:, 0], x0[:, ~deep][:, 0], x0[:, deep][:, 1], x0[:, ~deep][:, 1]])
    full, oi = _layout_invariance(lambda c, N_: engine.mpc_solve_batch(_cols(dA, c), _cols(dB, c), N_, pts=pts,
                                                                       S=S if c is None else len(c)), S, N, N + 9, seed=2)
    assert torch.equal(full["M_V"], full["V"].amax(0))
    g = {k: v[..., oi].cpu().numpy() for k, v in full.items()}
    dA_o, dB_o, _ = oracle_inputs(oi)
    pn = pts.cpu().numpy()
    for i in range(0, len(oi), 4):
        for p in range(4):
            _check_solve(N, *_model(A, B, dA_o, dB_o, i), Q, R, lo, hi, pn[p], g["V"][p, i], g["u0"][p, :, i],
                         g["flags"][p, i])
    # closed loops
    T = 8
    want = ("J_T", "flags", "n_active") + (("X", "U") if n <= 4 else ())
    for shared in (False, True):
        if shared:
            run = lambda c, N_: engine.simulate_batch(_cols(dA, c), _cols(dB, c), N_, T, x0_shared=pts[0],   # noqa
                                                      S=S if c is None else len(c), want=want)
        else:
            run = lambda c, N_: engine.simulate_batch(_cols(dA, c), _cols(dB, c), N_, T, x0=_cols(x0, c), want=want)  # noqa
        full, oi = _layout_invariance(run, S, N, N + 9, seed=3 + shared)
        g = {k: v[..., oi].cpu().numpy() for k, v in full.items()}
        dA_o, dB_o, x_o = oracle_inputs(oi)
        assert not np.any(g["flags"] & ~2)
        for i in range(0, len(oi), 3):
            xs = pn[0] if shared else x_o[:, i]
            _check_sim(T, N, *_model(A, B, dA_o, dB_o, i), Q, R, lo, hi, xs, A, B, g["J_T"][i],
                       g["X"][:, :, i].T if "X" in g else None, g["U"][:, :, i].T if "U" in g else None,
                       g["n_active"][i])


@pytest.mark.parametrize("n,m,N", K2_PAIRS)
def test_k2_references_and_polytope_multi_sample_launch(engine, n, m, N, monkeypatch):
    """K2 with non-zero references at the K2 pairs, and with a general input polytope at (4, 2), on multi-sample
    launches: layout invariance and the oracle."""
    import torch
    monkeypatch.setenv("LQMPC_K2_WAVES", "1")
    S = _sizes()[0]
    rng = np.random.default_rng(5000 + n)
    A, B, Q, R, lo, hi = _plant(rng, n, m, general=False, radius=(0.85, 0.95))
    engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
    dA, dB, d, deep = _batch(n, m, S, seed=10 + n)
    x0 = _scaled_states(A, B, Q, R, N, lo, hi, d, torch.where(deep, 5.0, 0.02))
    Nb = N + 9
    xr, ur = rng.normal(size=(n, Nb)) * 0.05, rng.normal(size=(m, Nb)) * 0.3 * np.min(hi)
    cpu = lambda t, oi: t[..., torch.as_tensor(oi, device="cuda")].cpu().numpy()   # noqa: E731
    with engine.references(xr, ur):
        full, oi = _layout_invariance(
            lambda c, N_: engine.mpc_solve_batch(_cols(dA, c), _cols(dB, c), N_, x0=_cols(x0, c)), S, N, Nb, seed=5)
    g = {k: v[..., oi].cpu().numpy() for k, v in full.items()}
    dA_o, dB_o, x_o = cpu(dA, oi), cpu(dB, oi), cpu(x0, oi)
    assert not np.any(g["flags"] & ~2)
    for i in range(0, len(oi), 2):
        _check_solve(N, *_model(A, B, dA_o, dB_o, i), Q, R, lo, hi, x_o[:, i], g["V"][0, i], g["u0"][0, :, i],
                     g["flags"][0, i], x_ref=xr, u_ref=ur)
    if (n, m) != (4, 2):
        return
    F = random_polytope(rng, m, 6, 0.15, 0.45)
    engine.set_problem(A, B, Q, R, Q, None, None, 10)
    engine.set_input_polytope(F)
    try:
        full, oi = _layout_invariance(
            lambda c, N_: engine.mpc_solve_batch(_cols(dA, c), _cols(dB, c), N_, x0=_cols(x0, c)), S, N, Nb, seed=6)
        sim, oj = _layout_invariance(
            lambda c, N_: engine.simulate_batch(_cols(dA, c), _cols(dB, c), N_, 5, x0=_cols(x0, c),
                                                want=("J_T", "U", "flags")), S, N, Nb, seed=7)
    finally:
        engine.set_input_polytope(None)
    g = {k: v[..., oi].cpu().numpy() for k, v in full.items()}
    dA_o, dB_o, x_o = cpu(dA, oi), cpu(dB, oi), cpu(x0, oi)
    n_act = 0
    for i in range(0, len(oi), 2):
        n_act += _check_solve(N, *_model(A, B, dA_o, dB_o, i), Q, R, None, None, x_o[:, i], g["V"][0, i],
                              g["u0"][0, :, i], g["flags"][0, i], F_u=F)[0]
    assert n_act > 0.2 * len(range(0, len(oi), 2))
    g = {k: v[..., oj].cpu().numpy() for k, v in sim.items()}
    dA_o, dB_o, x_o = cpu(dA, oj), cpu(dB, oj), cpu(x0, oj)
    for i in range(0, len(oj), 6):
        _check_sim(5, N, *_model(A, B, dA_o, dB_o, i), Q, R, None, None, x_o[:, i], A, B, g["J_T"][i], None,
                   g["U"][:, :, i].T, None, F_u=F)


@pytest.mark.parametrize("n,m", [(2, 1), (4, 2), (8, 2)])
@pytest.mark.parametrize("route", ["matrix_free", "dense", "dense_kron"])
def test_k3_multi_sample_launch(engine, n, m, route, monkeypatch):
    """K3 on a batch of >= 4 samples per thread of the dense route's capped grid (SMs x 8 CTAs): the matrix-free route
    (scalar weights), the dense route forced by LQMPC_K3_DENSE=1, and the dense route that non-scalar weights in the
    strict kron convention take. Per-sample e, M_V and states; layout invariance and the oracle."""
    import torch
    if route == "dense":
        monkeypatch.setenv("LQMPC_K3_DENSE", "1")
    else:
        monkeypatch.delenv("LQMPC_K3_DENSE", raising=False)
    S = _sizes()[1]
    rng = np.random.default_rng(6000 + n)
    A, B, Q, R, lo, hi = _plant(rng, n, m, general=False, radius=(0.2, 0.5))
    if route == "dense_kron":
        # non-scalar but well-conditioned weights: with a large eigenvalue spread of Q the reference's formulas have no
        # value (eta > 1 under a square root) on every sample, and xi / eta / bound would go unchecked
        Mq, Mr = rng.normal(size=(n, n)), rng.normal(size=(m, m))
        Q = Q + 0.1 * Q[0, 0] * (Mq @ Mq.T) / n
        R = R + 0.1 * R[0, 0] * (Mr @ Mr.T) / m
    engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
    dA, dB, d, deep = _batch(n, m, S, seed=20 + n)
    g = torch.Generator(device="cuda").manual_seed(30 + n)
    e = 10 ** (-4 + 2 * torch.rand(S, device="cuda", dtype=torch.float64, generator=g))
    MV = 0.05 + 2 * torch.rand(S, device="cuda", dtype=torch.float64, generator=g)
    x = d * torch.where(deep, 0.5, 1e-3)
    N = 8

    def run(c, N_):
        out = engine.bounds_batch(_cols(dA, c), _cols(dB, c), N_, _cols(e, c), _cols(e, c), _cols(MV, c), _cols(x, c),
                                  P3, 0.37, S=S if c is None else len(c), want_K=True, want_P=True)
        out["detail"] = torch.stack([out[f] for f in ("alpha", "beta", "xi", "eta", "bound", "min_H", "norm_Gamma")])
        return {k: out[k] for k in ("detail", "flags", "K", "P")}

    full, oi = _layout_invariance(run, S, N, N + 7, seed=8)
    oi_t = torch.as_tensor(oi, device="cuda")
    sub = engine.bounds_batch(dA[:, oi_t], dB[:, oi_t], N, e[oi_t], e[oi_t], MV[oi_t], x[:, oi_t], P3, 0.37,
                              want_K=True, want_P=True)
    for i, f in enumerate(("alpha", "beta", "xi", "eta", "bound", "min_H", "norm_Gamma")):
        assert _same_bits(sub[f], full["detail"][i, oi_t]), f
    gs = _np(sub)
    dA_o, dB_o, e_o, MV_o, x_o = (t[..., oi_t].cpu().numpy() for t in (dA, dB, e, MV, x))
    ok = sum(_check_bounds(gs, i, *_model(A, B, dA_o, dB_o, i), Q, R, lo, hi, N, e_o[i], MV_o[i], x_o[:, i], 0.37,
                           True) for i in range(len(oi)))
    assert ok > 0.2 * len(oi)                         # energy_decreasing defined on a good share of the samples


@pytest.mark.parametrize("n,m", [(5, 2), (12, 4)])
def test_warp_route_multi_sample_launch(engine, n, m):
    """The run-time-dimension route (one warp per sample, SMs x CTAs-per-SM grid) on a batch of >= 4 samples per
    launched warp: K1, K2 solves and closed loops (deep and tiny states interleaved), and K3 — layout invariance and
    the oracle."""
    import torch
    from oracle import np_batched as nb
    S = _sizes()[2]
    rng = np.random.default_rng(7000 + n)
    A, B, Q, R, lo, hi = _plant(rng, n, m, general=False, radius=(0.6, 0.9))
    engine.set_problem(A, B, Q, R, Q, lo, hi, 10)
    assert (n, m) not in engine.supported_dims()
    dA, dB, d, deep = _batch(n, m, S, seed=40 + n, e=0.003)
    cpu = lambda t, oi: t[..., torch.as_tensor(oi, device="cuda")].cpu().numpy()   # noqa: E731
    # K1
    full, oi = _layout_invariance(lambda c, N_: {k: v for k, v in engine.eval_batch(
        _cols(dA, c), _cols(dB, c), _cols(d, c), N_ - 2, N_, T=6, want=("J", "rho", "V_N", "J_T", "flags")).items()
        if k in ("J", "rho", "V_N", "J_T", "flags")}, S, 6, 11, seed=9)
    dA_o, dB_o, x_o = cpu(dA, oi), cpu(dB, oi), cpu(d, oi)
    ref = nb.eval_batch(A, B, Q, R, Q, nb.expert_matrix(A, B, Q, R, Q, 10), dA_o.T.reshape(-1, n, n),
                        dB_o.T.reshape(-1, n, m), x_o.T, 4, 6, T=6)
    g = {k: v[..., oi].cpu().numpy() for k, v in full.items()}
    assert np.array_equal((g["flags"] & 1) != 0, ref["unstable"]) and not np.any(g["flags"] & ~1)
    for k, kr in (("rho", "rho"), ("V_N", "Vn"), ("J_T", "JT"), ("J", "J")):
        assert relerr(g[k], ref[kr]) < TOL, k
    # K2
    N = 6
    x0 = _scaled_states(A, B, Q, R, N, lo, hi, d, torch.where(deep, 5.0, 0.02))
    full, oi = _layout_invariance(lambda c, N_: engine.mpc_solve_batch(_cols(dA, c), _cols(dB, c), N_, x0=_cols(x0, c)),
                                  S, N, N + 5, seed=10)
    g = {k: v[..., oi].cpu().numpy() for k, v in full.items()}
    dA_o, dB_o, x_o = cpu(dA, oi), cpu(dB, oi), cpu(x0, oi)
    n_act = 0
    for i in range(0, len(oi), 2):
        n_act += _check_solve(N, *_model(A, B, dA_o, dB_o, i), Q, R, lo, hi, x_o[:, i], g["V"][0, i], g["u0"][0, :, i],
                              g["flags"][0, i])[0]
    assert 0.3 * len(range(0, len(oi), 2)) < n_act < 0.7 * len(range(0, len(oi), 2))
    T = 5
    sim, oi = _layout_invariance(lambda c, N_: engine.simulate_batch(
        _cols(dA, c), _cols(dB, c), N_, T, x0=_cols(x0, c), want=("J_T", "U", "flags", "n_active")), S, N, N + 5,
        seed=11)
    g = {k: v[..., oi].cpu().numpy() for k, v in sim.items()}
    dA_o, dB_o, x_o = cpu(dA, oi), cpu(dB, oi), cpu(x0, oi)
    for i in range(0, len(oi), 6):
        _check_sim(T, N, *_model(A, B, dA_o, dB_o, i), Q, R, lo, hi, x_o[:, i], A, B, g["J_T"][i], None,
                   g["U"][:, :, i].T, g["n_active"][i])
    # K3
    x = d * 0.05
    full, oi = _layout_invariance(lambda c, N_: {k: v for k, v in engine.bounds_batch(
        _cols(dA, c), _cols(dB, c), N_, 2e-3, 2e-3, 0.5, _cols(x, c), P3, 0.37, S=S if c is None else len(c),
        want_K=True).items() if k in ("alpha", "beta", "xi", "eta", "bound", "flags", "K")}, S, 5, 7, seed=12)
    g = {k: v[..., oi].cpu().numpy() for k, v in full.items()}
    dA_o, dB_o, x_o = cpu(dA, oi), cpu(dB, oi), cpu(x, oi)
    from oracle import np_oracle as o
    for i in range(0, len(oi), 3):
        Ah, Bh = _model(A, B, dA_o, dB_o, i)
        K, _ = o.dlqr(Ah, Bh, Q, R)
        assert np.max(np.abs(g["K"][:, i].reshape(m, n) + K)) < TOL * max(1, np.max(np.abs(K)))
        bnd = o.energy_bound(Ah, Bh, Q, R, lo, hi, 5, 2e-3, 2e-3, x_o[:, i], P3)
        for f in ("alpha", "beta"):
            assert abs(g[f][i] - bnd[f]) <= TOL * abs(bnd[f]), f
        try:
            dec = o.energy_decreasing(Ah, Bh, Q, R, lo, hi, 5, 2e-3, 2e-3, -K, 0.5)
        except ValueError:
            assert g["flags"][i] & 512
            continue
        for f in ("xi", "eta"):
            assert abs(g[f][i] - dec[f]) <= TOL * abs(dec[f]), f


# ===================================================================================== C. host pipeline, every K1 build
@pytest.mark.parametrize("n,m,group", [(n, m, None) for n, m in ALL_DIMS] + [(8, 2, "0"), (8, 2, "2"), (8, 2, "4"),
                                                                            (6, 2, "0")])
def test_host_pipeline_every_k1_build(engine, n, m, group, monkeypatch):
    """eval_batch_host at every compiled pair (the lane-group K1 at n = 6, 8 and its other builds via LQMPC_K1_GROUP),
    S = 3 chunks + 37 so that the last chunk is ragged (its leading dimension is the chunk, not its sample count),
    nested and single horizons: bit for bit the device-resident eval_batch."""
    import torch
    from oracle import np_batched as nb
    if group is None:
        monkeypatch.delenv("LQMPC_K1_GROUP", raising=False)
    else:
        monkeypatch.setenv("LQMPC_K1_GROUP", group)
    A, B, Q, R = nb.synth_problem(n, m, seed=6)
    engine.set_problem(A, B, Q, R, Q, None, None, 30)
    chunk = 4096
    S = 3 * chunk + 37
    soa = nb.to_soa(*nb.synth_samples(n, m, S, seed=7, e=0.05))
    h = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in soa]
    for N_min, N_max in ((2, 6), (9, 9)):
        dev = engine.eval_batch(*soa, N_min, N_max)
        hp = engine.eval_batch_host(h[0], h[1], h[2], N_min, N_max, chunk=chunk)
        for k in ("J", "rho", "ratio", "flags"):
            assert np.array_equal(hp[k].numpy(), dev[k].cpu().numpy(), equal_nan=k != "flags"), (N_min, N_max, k)
