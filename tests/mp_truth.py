"""TEST INFRASTRUCTURE ONLY — extended-precision (mpmath, 50 digits) arbitration of the hot path.

Where the CUDA engine and the float64 numpy oracle disagree by more than north_star's 1e-9, neither is trusted: the
quantity is recomputed here in 50-digit arithmetic from the SAME float64 inputs and both are measured against it.
This is what turns "the comparison is ill-conditioned" from an assertion into a measured statement:
  * `k1_truth`   Riccati gain of horizon N on (A+dA, B+dB), closed loop on (A, B), J_inf by a direct solve of the
                 discrete Lyapunov equation (vec form), rho by mpmath's eigenvalue solver, V_N — the quantities of
                 utils_class.py:48-91, 245-285 for an inactive input set;
  * `qp_truth`   the box-constrained condensed QP of utils_class.py:59-88 solved on a GIVEN active set in 50 digits,
                 with the KKT sign conditions re-checked there (so the active set is certified, not assumed).
Slow (pure Python): meant for a handful of samples.
"""
from __future__ import annotations

import mpmath as mp
import numpy as np

mp.mp.dps = 50


def _M(a):
    a = np.atleast_2d(np.asarray(a, dtype=float))
    return mp.matrix(a.tolist())


def _riccati_gain(Ah, Bh, Q, R, Pt, N):
    P = Pt.copy()
    K = None
    for _ in range(N):
        G = R + Bh.T * P * Bh
        H = Bh.T * P * Ah
        K = -mp.lu_solve(G, H)
        P = Q + Ah.T * P * Ah + H.T * K
        P = (P + P.T) / 2
    return K, P


def k1_truth(A, B, Q, R, Pt, dA, dB, x0, N):
    """Returns dict(J, rho, Vn, K0) as Python floats / arrays rounded from 50-digit results."""
    A, B, Q, R, Pt = _M(A), _M(B), _M(Q), _M(R), _M(Pt)
    n, m = A.rows, B.cols
    Ah, Bh = A + _M(dA), B + _M(np.asarray(dB, dtype=float).reshape(n, m))
    x = mp.matrix([mp.mpf(float(v)) for v in np.asarray(x0, dtype=float).reshape(-1)])
    K, P = _riccati_gain(Ah, Bh, Q, R, Pt, N)
    Acl = A + B * K
    W = Q + K.T * R * K
    ev, _ = mp.eig(Acl)
    rho = max(abs(e) for e in ev)
    out = {"rho": float(rho), "Vn": float((x.T * P * x)[0]),
           "K0": np.array([[float(K[i, j]) for j in range(n)] for i in range(m)])}
    if rho >= 1:
        out["J"] = float("inf")
        return out
    # S = W + Acl' S Acl  <=>  (I - Acl' (x) Acl') vec(S) = vec(W)   (row-major vec)
    AT = Acl.T
    big = mp.eye(n * n)
    for i in range(n):
        for j in range(n):
            for k in range(n):
                for l in range(n):
                    big[i * n + j, k * n + l] -= AT[i, k] * AT[j, l]
    vw = mp.matrix([W[i, j] for i in range(n) for j in range(n)])
    vs = mp.lu_solve(big, vw)
    S = mp.matrix(n, n)
    for i in range(n):
        for j in range(n):
            S[i, j] = vs[i * n + j]
    out["J"] = float((x.T * S * x)[0])
    return out


def j_condition_bound(rho):
    """Relative rounding-error allowance for J_inf = x0' S x0 in float64: perturbing A_cl by one rounding error u moves
    rho by ~u and J ~ sum rho^(2k) by dJ/J ~ 2 rho d(rho) / (1 - rho^2), i.e. the relative condition number is
    ~rho / (1 - rho); 16 u rho/(1 - rho) allows a handful of such errors. It exceeds 1e-9 only within 1.8e-6 of the
    stability boundary."""
    u = 2.0 ** -53
    return max(1e-9, 16.0 * u * rho / max(1.0 - rho, 1e-300))


def qp_truth(N, A, B, Q, R, P, lo, hi, x0, active_lo, active_hi):
    """Condensed QP min z'Hz + 2g'z (+ c0 + x0'Qx0) with the components in `active_lo` / `active_hi` clamped, solved in
    50 digits. Returns (u0, V, certified): certified = every free component strictly inside its bounds (to 1e-30) and
    every clamped one with the right multiplier sign."""
    A, B, Q, R, P = _M(A), _M(B), _M(Q), _M(R), _M(P)
    n, m = A.rows, B.cols
    nz = N * m
    # Gamma rows for x_1..x_N and Phi
    Gam = mp.zeros(N * n, nz)
    AB = B.copy()
    for d in range(N):
        for j in range(N - d):
            i = j + d
            for r in range(n):
                for c in range(m):
                    Gam[i * n + r, j * m + c] = AB[r, c]
        AB = A * AB
    x = mp.matrix([mp.mpf(float(v)) for v in np.asarray(x0, dtype=float).reshape(-1)])
    f = mp.zeros(N * n, 1)
    Mk = A.copy()
    for k in range(N):
        v = Mk * x
        for r in range(n):
            f[k * n + r] = v[r]
        Mk = A * Mk
    Wb = mp.zeros(N * n, N * n)
    for k in range(N):
        blk = P if k == N - 1 else Q
        for r in range(n):
            for c in range(n):
                Wb[k * n + r, k * n + c] = blk[r, c]
    H = Gam.T * Wb * Gam
    for k in range(N):
        for r in range(m):
            for c in range(m):
                H[k * m + r, k * m + c] += R[r, c]
    g = Gam.T * Wb * f
    c0 = (f.T * Wb * f)[0] + (x.T * Q * x)[0]
    lo_t = [mp.mpf(float(lo[j % m])) for j in range(nz)]
    hi_t = [mp.mpf(float(hi[j % m])) for j in range(nz)]
    z = mp.zeros(nz, 1)
    fixed = {}
    for j in active_lo:
        fixed[int(j)] = lo_t[int(j)]
    for j in active_hi:
        fixed[int(j)] = hi_t[int(j)]
    free = [j for j in range(nz) if j not in fixed]
    for j, v in fixed.items():
        z[j] = v
    if free:
        Hff = mp.matrix(len(free), len(free))
        rhs = mp.matrix(len(free), 1)
        for a, ja in enumerate(free):
            acc = -g[ja]
            for jb, v in fixed.items():
                acc -= H[ja, jb] * v
            rhs[a] = acc
            for b, jb in enumerate(free):
                Hff[a, b] = H[ja, jb]
        zf = mp.lu_solve(Hff, rhs)
        for a, ja in enumerate(free):
            z[ja] = zf[a]
    grad = 2 * (H * z + g)
    ok = True
    for j in free:
        if not (lo_t[j] - mp.mpf(10) ** -30 <= z[j] <= hi_t[j] + mp.mpf(10) ** -30):
            ok = False
    for j in active_lo:
        if grad[int(j)] < -mp.mpf(10) ** -30:
            ok = False
    for j in active_hi:
        if grad[int(j)] > mp.mpf(10) ** -30:
            ok = False
    V = (z.T * H * z)[0] + 2 * (g.T * z)[0] + c0
    return np.array([float(z[j]) for j in range(m)]), float(V), ok


# ------------------------------------------------------------------------------------------------ longdouble (n = 32)
def _ld_solve(G, H):
    """Gaussian elimination with partial pivoting in numpy longdouble (x87 80-bit: 64-bit mantissa)."""
    G = G.copy()
    H = H.copy()
    k = G.shape[0]
    for c in range(k):
        p = c + int(np.argmax(np.abs(G[c:, c])))
        if p != c:
            G[[c, p]] = G[[p, c]]
            H[[c, p]] = H[[p, c]]
        for r in range(c + 1, k):
            f = G[r, c] / G[c, c]
            G[r, c:] -= f * G[c, c:]
            H[r] -= f * H[c]
    X = np.zeros_like(H)
    for r in range(k - 1, -1, -1):
        X[r] = (H[r] - G[r, r + 1:] @ X[r + 1:]) / G[r, r]
    return X


def _k1_ld(A, B, Q, R, Pt, dA, dB, x0, N):
    ld = np.longdouble
    A, B, Q, R, P = (np.asarray(a, dtype=ld) for a in (A, B, Q, R, Pt))
    n, m = B.shape
    Ah, Bh = A + np.asarray(dA, dtype=ld), B + np.asarray(dB, dtype=ld).reshape(n, m)
    x = np.asarray(x0, dtype=ld).reshape(n)
    K = None
    for _ in range(N):
        G = R + Bh.T @ P @ Bh
        H = Bh.T @ P @ Ah
        K = -_ld_solve(G, H)
        P = Q + Ah.T @ P @ Ah + H.T @ K
        P = (P + P.T) / 2
    Acl = A + B @ K
    W = Q + K.T @ R @ K
    rho = float(np.max(np.abs(np.linalg.eigvals(Acl.astype(np.float64)))))
    out = {"rho": rho, "Vn": float(x @ P @ x)}
    if rho >= 1:
        out["J"] = float("inf")
        return out
    S, M = W.copy(), Acl.copy()
    for _ in range(80):
        T = M.T @ S @ M
        S = S + T
        if float(np.max(np.abs(T))) <= 1e-24 * float(np.max(np.abs(S))):
            break
        M = M @ M
    out["J"] = float(x @ S @ x)
    return out


def k1_truth_ld(A, B, Q, R, Pt, dA, dB, x0, N, delta=1e-13, seed=0):
    """Extended-precision (longdouble) K1 values for larger n, plus the MEASURED relative condition number of each
    value with respect to the sample: kappa_X = |X(dA (1 + delta r)) - X(dA)| / (|X| delta), r ~ U[-1, 1] entrywise.
    A backward-stable float64 evaluation cannot be expected to do better than ~kappa u."""
    base = _k1_ld(A, B, Q, R, Pt, dA, dB, x0, N)
    rng = np.random.default_rng(seed)
    pert = np.asarray(dA, dtype=np.longdouble) * (1 + np.longdouble(delta) * rng.uniform(-1, 1, size=np.shape(dA)))
    other = _k1_ld(A, B, Q, R, Pt, pert, dB, x0, N)
    for k in ("J", "Vn", "rho"):
        if np.isfinite(base[k]) and np.isfinite(other[k]) and base[k] != 0:
            base["kappa_" + k] = abs(other[k] - base[k]) / (abs(base[k]) * delta)
        else:
            base["kappa_" + k] = float("inf")
    return base


# ------------------------------------------------------------------------------------------------ K3 (bounds)
# Names of the 31 fields of lqmpc_bounds_batch's detail table, in its order.
BOUND_FIELDS = ['alpha', 'beta', 'xi', 'eta', 'bound', 'E_psi', 'E_u', 'E_psi_u', 'theta_u', 'theta_x_u', 'C_K',
                'rho_K', 'gamma', 'rho_gamma', 'L_V', 'N_0', 'omega_N1', 'omega_N0d5', 'err_th', 'N_min', 'h',
                'epsilon_K', 'norm_A', 'norm_B', 'norm_K', 'norm_Gamma', 'norm_Phi', 'min_H', 'rho_cl', 'bar_u',
                'bar_d_u']
# the matrix quantities the scalar formulas start from (what bounds_formulas receives from the matrix part)
K3_INTERMEDIATES = ('fA', 'fB', 'nK', 'eps_K', 'rho_cl', 'nPhi', 'cmax', 'min_H')
_NAN = mp.mpf('nan')


def _rows(M):
    return [[M[i, j] for j in range(M.cols)] for i in range(M.rows)]


def _sym_extremes(M):
    ev = mp.eigsy(M, eigvals_only=True)
    ev = sorted(ev[i] for i in range(M.rows))
    return ev[0], ev[-1]


def _norm2(M):
    return mp.sqrt(max(_sym_extremes(M.T * M)[1], mp.mpf(0)))


def _gram_blocks(Ah, Bh, N):
    """G_d = A^d B, d = 0..N-1, as n x m mp matrices."""
    G, out = Bh.copy(), []
    for _ in range(N):
        out.append(G)
        G = Ah * G
    return out


def gram_truth(Ah, Bh, Q, R, N, strict_reference=True):
    """lambda_max(Gamma'Gamma), lambda_min(H^), lambda_max(H^) of horizon N by mp.eigsy on the ASSEMBLED 50-digit
    matrices: Gamma of utils.py:145-174 (block (t, j) = A^(t-1-j) B for t > j, rows x_0..x_N) and
    H^ = barR + Gamma' barQ Gamma with the literal kron(Q, I_{N+1}), kron(R, I_N) ordering of utils.py:317-318
    (strict_reference) or the time-major block-diagonal weights. Scalar weights give the same H^ in both."""
    Ah, Bh, Q, R = _M(Ah), _M(Bh), _M(Q), _M(R)
    n, m = Bh.rows, Bh.cols
    k, rows = N * m, (N + 1) * n
    Gs = _gram_blocks(Ah, Bh, N)
    Gam = mp.zeros(rows, k)
    for j in range(N):
        for t in range(j + 1, N + 1):
            G = Gs[t - 1 - j]
            for r in range(n):
                for s in range(m):
                    Gam[t * n + r, j * m + s] = G[r, s]
    GtG = Gam.T * Gam
    cmin, cmax = _sym_extremes(GtG)
    scalar = all(Q[i, j] == (Q[0, 0] if i == j else 0) for i in range(n) for j in range(n)) and \
        all(R[i, j] == (R[0, 0] if i == j else 0) for i in range(m) for j in range(m))
    if scalar:                           # H^ = r I + q Gamma'Gamma in either ordering
        hmin, hmax = R[0, 0] + Q[0, 0] * cmin, R[0, 0] + Q[0, 0] * cmax
    else:
        bQ, bR = mp.zeros(rows, rows), mp.zeros(k, k)
        for a in range(rows):
            for b in range(rows):
                if strict_reference:
                    if a % (N + 1) == b % (N + 1):
                        bQ[a, b] = Q[a // (N + 1), b // (N + 1)]
                elif a // n == b // n:
                    bQ[a, b] = Q[a % n, b % n]
        for c in range(k):
            for d in range(k):
                if strict_reference:
                    if c % N == d % N:
                        bR[c, d] = R[c // N, d // N]
                elif c // m == d // m:
                    bR[c, d] = R[c % m, d % m]
        H = bR + Gam.T * bQ * Gam
        hmin, hmax = _sym_extremes((H + H.T) / 2)
    return {"cmax": cmax, "min_H": hmin, "max_H": hmax, "cond_H": hmax / hmin}


def dare_truth(Ah, Bh, Q, R, tol=mp.mpf(10) ** -45, max_iter=20000):
    """Stabilising DARE solution by Riccati iteration from P = Q to convergence in 50 digits, and the gain
    K = (R + B'PB)^-1 B'PA of control.dlqr (u = -Kx)."""
    Ah, Bh, Q, R = _M(Ah), _M(Bh), _M(Q), _M(R)
    P = Q.copy()
    for _ in range(max_iter):
        G = R + Bh.T * P * Bh
        H = Bh.T * P * Ah
        Pn = Q + Ah.T * P * Ah - H.T * (mp.inverse(G) * H)
        Pn = (Pn + Pn.T) / 2
        d = mp.mnorm(Pn - P, 1)
        P = Pn
        if d <= tol * mp.mnorm(P, 1):
            break
    else:
        raise RuntimeError("Riccati iteration did not converge")
    K = mp.inverse(R + Bh.T * P * Bh) * (Bh.T * P * Ah)
    return K, P


def _eig_condition(M):
    """(rho(M), relative condition of rho): |d rho| <= kappa * ||dM||_2 / rho * rho ... i.e. kappa = ||M|| / (rho |y'x|)
    for the dominant eigenvalue with unit left / right eigenvectors y, x (Wilkinson's 1 / |y'x|), maximised over the
    eigenvalues of largest modulus."""
    ev, ER = mp.eig(M)
    EL = mp.inverse(ER)              # rows: left eigenvectors (y' = row of ER^-1, y'x = 1)
    rho = max(abs(e) for e in ev)
    nM = _norm2(M)
    kap = mp.mpf(1)
    for i, e in enumerate(ev):
        if abs(e) < rho * (1 - mp.mpf(10) ** -20):
            continue
        x = ER[:, i]
        y = EL[i, :]
        nx = mp.sqrt(sum(abs(x[r]) ** 2 for r in range(M.rows)))
        ny = mp.sqrt(sum(abs(y[r]) ** 2 for r in range(M.rows)))
        kap = max(kap, nx * ny * nM / max(rho, mp.mpf(10) ** -40))
    return rho, kap


def _formulas(c, q, N0_fixed=None):
    """bounds_formulas / np_oracle's energy_decreasing, energy_bound in mp from the constants c and the matrix
    quantities q. Out-of-domain log / sqrt arguments give NaN (IEEE semantics: the reference raises there).
    Returns (fields, edge arguments)."""
    nan = _NAN
    maxQ, minQ, maxR, minR = c["maxQ"], c["minQ"], c["maxR"], c["minR"]
    N, e_A, e_B, M_V = c["N"], c["e_A"], c["e_B"], c["M_V"]
    fA, fB, nK, eps, rho_cl, nPhi, cmax, min_H = (q[k] for k in K3_INTERMEDIATES)
    bu, bdu, nx2 = c["bu"], c["bdu"], c["nx2"]
    ratioQ = maxQ / minQ
    o = {"bar_u": bu, "bar_d_u": bdu, "norm_A": fA, "norm_B": fB, "norm_K": nK, "epsilon_K": eps,
         "rho_cl": rho_cl, "norm_Phi": nPhi, "norm_Gamma": mp.sqrt(max(cmax, 0)), "min_H": min_H}
    nG = o["norm_Gamma"]
    rho_K = (rho_cl + mp.mpf("0.4")) ** 2
    C_K = (1 + maxR * nK ** 2 / minQ) * max(mp.mpf(1), ratioQ * mp.mpf("1.21"))
    gam = C_K / (1 - rho_K) if rho_K != 1 else nan
    rho_g = (gam - 1) / gam
    o.update(C_K=C_K, rho_K=rho_K, gamma=gam, rho_gamma=rho_g)
    mv_eps = M_V / eps if mp.isfinite(eps) else mp.mpf(0)
    L_V = max(gam, mv_eps) if not mp.isnan(gam) else nan
    N0_arg = max(mp.mpf(0), mv_eps - gam) if not mp.isnan(gam) else nan
    N_0 = (mp.ceil(N0_arg) if N0_fixed is None else N0_fixed) if not mp.isnan(N0_arg) else nan
    o.update(L_V=L_V, N_0=N_0)
    fA2 = fA * fA
    G_A = mp.mpf(N - 1) if fA == 1 else (1 - fA ** (2 * (N - 1))) / (1 - fA2)
    term = 1 + fA2 * ratioQ
    arg1 = fA2 * ratioQ * gam
    log_ok = (arg1 > 0) and (rho_g > 0)
    nmin_arg = N_0 - mp.log(arg1) / mp.log(rho_g) if log_ok and rho_g != 1 else nan
    o["N_min"] = mp.ceil(nmin_arg) if not mp.isnan(nmin_arg) else nan
    fApow = fA ** (2 * N - 2)
    rg_pow = rho_g ** (N - N_0) if not (mp.isnan(rho_g) or mp.isnan(N_0)) else nan
    w1 = maxQ * (term * fApow + G_A)
    decay = maxQ * fApow * gam * rg_pow
    w05_a = maxQ * (L_V - 1) * G_A
    sq = lambda v: mp.sqrt(v) if (not mp.isnan(v)) and v >= 0 else nan   # noqa: E731
    w05 = sq(w05_a) + mp.mpf("0.5") * term * sq(decay)
    eta = (term - 1) * gam * rg_pow
    disc = w05 * w05 + w1 * (1 - eta)
    err_r = (sq(disc) - w05) / w1
    o.update(omega_N1=w1, omega_N0d5=w05, eta=eta, err_th=err_r * err_r)
    h = e_A * e_A / minQ + e_B * e_B / minR
    xi = h * w1 + 2 * mp.sqrt(h) * w05
    o.update(h=h, xi=xi)
    nx = mp.sqrt(nx2)
    eAfA, eBfB = e_A + fA, e_B + fB
    s_in = s_out = bgx = bgu = bgu_in = mp.mpf(0)
    for i in range(N + 1):
        fpi = fA ** i
        gx1 = eAfA ** i - fpi
        gu1 = eBfB * gx1 + e_B * fpi
        s_out += (s_in + gx1 * gx1) * (nx * nx + i * bu)
        s_in += gu1 * gu1
        if i >= 1:
            bgx += gx1
        if i < N:
            bgu_in += gu1
            bgu += bgu_in
    E_psi = maxQ * s_out
    theta_u = maxQ * (2 * nG * bgu + bgu * bgu)
    theta_xu = maxQ * (nG * bgx + nPhi * bgu + bgx * bgu)
    bar_theta = mp.sqrt(N * bu) * theta_u + nx * theta_xu
    cand = min(mp.sqrt(N * bdu), bar_theta / min_H)
    E_u = maxR * cand * cand
    E_psi_u = maxQ / maxR * (nG + bgu) ** 2 * E_u
    o.update(E_psi=E_psi, E_u=E_u, E_psi_u=E_psi_u, theta_u=theta_u, theta_x_u=theta_xu)
    sp, su, spu = mp.sqrt(E_psi), mp.sqrt(E_u), mp.sqrt(E_psi_u)
    p0, p1, p2 = c["p"]
    alpha = max(p0 * sp + p2 * spu + p0 * sp * p2 * spu, p1 * su)
    beta = (1 + p0 * sp) * ((1 / p2) * spu + E_psi_u) + (1 / p1) * su + E_u + (1 / p0) * sp + E_psi
    den = 1 - xi - eta
    o.update(alpha=alpha, beta=beta, bound=(alpha * c["V_expert"] + beta) / den)
    edges = {"den": den, "arg1": arg1, "rho_gamma": rho_g, "one_minus_rho_K": 1 - rho_K, "sqrt_w05": w05_a,
             "sqrt_decay": decay, "sqrt_disc": disc, "N0_arg": N0_arg, "Nmin_arg": nmin_arg}
    return o, edges


def k3_prefix_truth(A_hat, B_hat, Q, R, lo, hi, K=None):
    """The horizon-independent part of k3_truth (one per model): gain, norms, local_radius, rho(A^ + B^K) and its
    eigenvalue condition number."""
    Ah, Bh, Qm, Rm = _M(A_hat), _M(B_hat), _M(Q), _M(R)
    n, m = Bh.rows, Bh.cols
    lo, hi = np.asarray(lo, dtype=float).reshape(m), np.asarray(hi, dtype=float).reshape(m)
    if K is None:
        Km = -dare_truth(A_hat, B_hat, Q, R)[0]
    else:
        Km = _M(np.asarray(K, dtype=float).reshape(m, n))
    qmin, qmax = _sym_extremes(Qm)
    rmin, rmax = _sym_extremes(Rm)
    Qi = mp.inverse(Qm)
    amax = mp.mpf(0)
    for j in range(m):
        kq = (Km[j, :] * Qi * Km[j, :].T)[0]
        for b in (lo[j], hi[j]):
            if np.isfinite(b):
                amax = max(amax, kq / mp.mpf(float(b)) ** 2)
    rho_cl, kap_rho = _eig_condition(Ah + Bh * Km)
    return {"Ah": Ah, "K": Km, "maxQ": qmax, "minQ": qmin, "maxR": rmax, "minR": rmin,
            "bu": sum(max(mp.mpf(float(lo[j])) ** 2, mp.mpf(float(hi[j])) ** 2) for j in range(m)),
            "bdu": sum((mp.mpf(float(hi[j])) - mp.mpf(float(lo[j]))) ** 2 for j in range(m)),
            "fA": _norm2(Ah), "fB": _norm2(Bh), "nK": _norm2(Km), "eps_K": 1 / amax if amax > 0 else mp.inf,
            "rho_cl": rho_cl, "rho_cl_condition": kap_rho}


def k3_truth(A_hat, B_hat, Q, R, lo, hi, N, e_A, e_B, M_V, x, p, V_expert, strict_reference, K=None, gram=None,
             prefix=None, kappa=True):
    """50-digit K3 of one sample from the same float64 inputs: every field of BOUND_FIELDS (mp values; NaN where the
    reference raises before producing it), plus
      'K'       the terminal gain used (u = +Kx: -K_dlqr of the 50-digit DARE unless K is given),
      'edges'   signed edge arguments: den = 1 - xi - eta, arg1 and rho_gamma of math.log, 1 - rho_K, the three
                math.sqrt arguments (omega_N0d5's two, err_th's), and the arguments of N_0's and N_min's ceil,
      'raises'  True / False: a log / sqrt argument out of domain or a division by 1 - rho_K = 0 (the reference
                raises ValueError / ZeroDivisionError); decided in 50 digits,
      'kappa'   per field, the relative condition factor with respect to the matrix quantities K3_INTERMEDIATES
                (sum over them of |d ln field / d ln q|, each weighted by the relative accuracy its float64
                computation can reach in units of u: 1 for norms and Gram extremes, the eigenvalue condition
                number for rho_cl), N_0 / N_min held at their ceil,
      'cond_H'  cond(H^), 'ceil_dist' the distance of N_0's and N_min's ceil arguments from the integers.
    `gram`: precomputed gram_truth of (A_hat, B_hat, Q, R, N, strict_reference), or False to skip the Gram extremes
    (alpha, beta, bound and the fields behind them are then NaN); `prefix`: precomputed k3_prefix_truth of the model;
    kappa=False skips the condition factors."""
    pre = prefix if prefix is not None else k3_prefix_truth(A_hat, B_hat, Q, R, lo, hi, K)
    Ah = pre["Ah"]
    n = Ah.rows
    xv = [mp.mpf(float(v)) for v in np.asarray(x, dtype=float).reshape(n)]
    c = {"maxQ": pre["maxQ"], "minQ": pre["minQ"], "maxR": pre["maxR"], "minR": pre["minR"], "N": int(N),
         "e_A": mp.mpf(float(e_A)), "e_B": mp.mpf(float(e_B)), "M_V": mp.mpf(float(M_V)), "bu": pre["bu"],
         "bdu": pre["bdu"], "nx2": sum(v * v for v in xv),
         "p": [mp.mpf(float(v)) for v in np.asarray(p, dtype=float).reshape(3)], "V_expert": mp.mpf(float(V_expert))}
    Pg = mp.eye(n)
    Mt = mp.eye(n)
    for _ in range(int(N)):
        Mt = Ah * Mt
        Pg += Mt.T * Mt
    if gram is False:                    # energy_decreasing only: the Gram extremes enter alpha, beta, bound alone
        g = {"cmax": _NAN, "min_H": _NAN, "cond_H": _NAN}
    else:
        g = gram if gram is not None else gram_truth(A_hat, B_hat, Q, R, int(N), strict_reference)
    q = {"fA": pre["fA"], "fB": pre["fB"], "nK": pre["nK"], "eps_K": pre["eps_K"], "rho_cl": pre["rho_cl"],
         "nPhi": mp.sqrt(_sym_extremes(Pg)[1]), "cmax": g["cmax"], "min_H": g["min_H"]}
    kap_rho = pre["rho_cl_condition"]
    out, edges = _formulas(c, q)
    weight = {k: mp.mpf(1) for k in K3_INTERMEDIATES}
    weight["rho_cl"] = kap_rho
    kappa = {f: mp.mpf(0) for f in BOUND_FIELDS}
    delta = mp.mpf(10) ** -25
    for k in (K3_INTERMEDIATES if kappa else ()):
        if not mp.isfinite(q[k]) or q[k] == 0:
            continue
        qp = dict(q)
        qp[k] = q[k] * (1 + delta)
        op, _ = _formulas(c, qp, N0_fixed=out["N_0"])
        for f in BOUND_FIELDS:
            if f in ("N_0", "N_min"):
                continue
            a, b = out[f], op[f]
            if mp.isfinite(a) and mp.isfinite(b) and a != 0:
                kappa[f] += weight[k] * abs((b - a) / a) / delta
    raises = bool((not (edges["arg1"] > 0)) or (not (edges["rho_gamma"] > 0)) or edges["one_minus_rho_K"] == 0
                  or edges["sqrt_w05"] < 0 or edges["sqrt_decay"] < 0 or edges["sqrt_disc"] < 0)

    def ceil_dist(v):
        if not mp.isfinite(v):
            return mp.inf
        return abs(v - mp.nint(v))
    return {"fields": out, "K": pre["K"], "edges": edges, "raises": raises, "kappa": kappa, "cond_H": g["cond_H"],
            "ceil_dist": {"N_0": ceil_dist(edges["N0_arg"]) if edges["N0_arg"] > 0 else mp.inf,
                          "N_min": ceil_dist(edges["Nmin_arg"])}, "q": q, "rho_cl_condition": kap_rho}


def k3_expected_flags(t, margin):
    """What bits 32 (BOUND_INVALID) and 512 (DOMAIN_ERROR) of the kernel must be for the truth t, or None where the
    sample lies within `margin` (relative) of an edge that decides the bit: (bit32, bit512) entries of True / False /
    None. Bit 512: a log or sqrt argument out of domain, or 1 - rho_K = 0 (the kernel then divides by zero and
    rho_gamma is NaN). Bit 32: not (1 - xi - eta > 0), NaN included (an out-of-domain sqrt inside xi)."""
    e = t["edges"]
    f = t["fields"]

    def side(v, scale):
        """+1 clearly inside the domain (v > 0), -1 clearly outside, 0 within the margin; NaN counts as outside."""
        if mp.isnan(v) or v == 0:        # an exact zero is decisive: log(0), a division by zero
            return -1
        if abs(v) <= margin * scale:
            return 0
        return 1 if v > 0 else -1
    one = mp.mpf(1)
    gam_scale = abs(f["gamma"]) if mp.isfinite(f["gamma"]) else one
    sides = [side(e["one_minus_rho_K"], mp.mpf(1)), side(e["arg1"], abs(e["arg1"]) / max(gam_scale, one) + margin),
             side(e["rho_gamma"], one / max(gam_scale, one))]
    for k in ("sqrt_w05", "sqrt_decay"):
        sides.append(side(e[k], abs(e[k]) if mp.isnan(e[k]) else max(abs(e[k]), mp.mpf(10) ** -300)) if e[k] != 0
                     else 1)
    disc_scale = f["omega_N0d5"] ** 2 + abs(f["omega_N1"] * (1 - f["eta"])) if mp.isfinite(f["eta"]) else one
    sides.append(side(e["sqrt_disc"], disc_scale) if not mp.isnan(e["sqrt_disc"]) else 1)
    # (the first three are log / division arguments: out of domain at 0 as well; the sqrt arguments only below 0)
    b512 = True if any(s < 0 for s in sides) else (False if all(s > 0 for s in sides) else None)
    if mp.isnan(e["den"]):
        b32 = True if b512 else None
    else:
        s = side(e["den"], 1 + abs(f["xi"]) + abs(f["eta"]))
        b32 = None if s == 0 else (s < 0)
    return b32, b512
