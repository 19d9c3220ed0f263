"""Host-side sample generation (SURVEY 8a rows a8/a9): model-error grids and synthetic problem/sample sets.

The reference's sampler is unseeded (`random.uniform`, utils.py:774) and forces the first N_matrix draws of every
level onto the norm boundary by rejection with np.isclose (utils.py:803,814) — a very low-yield loop. Here:
  * `reference_random_matrix(..., literal=True)` keeps that exact procedure (unseeded unless `rng` is given);
  * the default draws the same distribution for the interior samples and *rescales* the boundary ones onto
    ||.|| = bound (documented deviation: same support, no rejection loop), from a seeded Philox stream.
Layouts follow the reference's files: error_A (n, n, 5*N_matrix, n_err), error_B (n, m, 5*N_matrix, n_err).
"""
from __future__ import annotations

import random as _random

import numpy as np

_PHILOX_STREAM = 0x4C514D50   # "LQMP"


def _norm(M, norm_type):
    return np.linalg.norm(M) if norm_type == 'f' else np.linalg.norm(M, ord=2)


def reference_random_matrix(M, N_matrix, norm_bound, norm_type, rng=None, literal=False):
    """utils.py:779-823. Returns (rows, cols, 5*N_matrix)."""
    if norm_type not in ('f', '2'):
        return np.zeros([M.shape[0], M.shape[1], 5 * N_matrix])   # the reference leaves zeros for other types
    r, c = M.shape
    out = np.zeros([r, c, 5 * N_matrix])
    if literal:
        uni = (lambda: np.array([[_random.uniform(-norm_bound, norm_bound) for _ in range(c)] for _ in range(r)])) \
            if rng is None else (lambda: rng.uniform(-norm_bound, norm_bound, size=(r, c)))
        k = 0
        while k < N_matrix:
            T = uni()
            if np.isclose(_norm(T, norm_type), norm_bound):
                out[:, :, k] = T
                k += 1
        while k < 5 * N_matrix:
            T = uni()
            if _norm(T, norm_type) <= norm_bound:
                out[:, :, k] = T
                k += 1
        return out
    rng = np.random.default_rng() if rng is None else rng
    # vectorised: candidates are drawn in blocks (same stream order as one-by-one draws) and classified at once
    ordv = 'fro' if norm_type == 'f' else 2
    k, total = 0, 5 * N_matrix
    while k < total:
        blk = max(64, 4 * (total - k))
        T = rng.uniform(-norm_bound, norm_bound, size=(blk, r, c))
        nv = np.linalg.norm(T, ord=ordv, axis=(1, 2))
        if k < N_matrix:                      # boundary samples: rescale onto ||.|| = bound (no isclose rejection)
            ok = np.flatnonzero(nv > 0)[:N_matrix - k]
            out[:, :, k:k + len(ok)] = np.moveaxis(T[ok] * (norm_bound / nv[ok])[:, None, None], 0, -1)
            k += len(ok)
            if k < N_matrix:
                continue
            T, nv = T[ok[-1] + 1:], nv[ok[-1] + 1:]     # the rest of the block feeds the interior samples
        ok = np.flatnonzero(nv <= norm_bound)[:total - k]
        out[:, :, k:k + len(ok)] = np.moveaxis(T[ok], 0, -1)
        k += len(ok)
    return out


def seeded_error_grids(n, m, error_vec, N_matrix, norm_type, seed=20240522):
    """cfg-sweep grids (SURVEY 8d.3): (n,n,5*N_matrix,n_err) and (n,m,5*N_matrix,n_err) from Philox(seed)."""
    rng = np.random.Generator(np.random.Philox(key=[seed, _PHILOX_STREAM]))
    eA = np.zeros([n, n, 5 * N_matrix, len(error_vec)])
    eB = np.zeros([n, m, 5 * N_matrix, len(error_vec)])
    for i, e in enumerate(error_vec):
        eA[:, :, :, i] = reference_random_matrix(np.zeros((n, n)), N_matrix, e, norm_type, rng)
        eB[:, :, :, i] = reference_random_matrix(np.zeros((n, m)), N_matrix, e, norm_type, rng)
    return eA, eB


def device_error_grids(engine, n, m, error_vec, N_matrix, norm_type, seed=20240522, j_first=0, N_sys=None,
                        allow_projected=False, return_stats=False):
    """cfg-sweep grids generated in HBM by K6 (`lqmpc_sample_error_grid`): the counter-based restatement of
    error_matrix_generator (utils.py:826-847). Returns SoA device tensors dA [n*n][N_sys*n_err], dB [n*m][N_sys*n_err]
    (sample s = j*n_err + i) — reshape(n, n|m, N_sys, n_err) gives the reference's file layout. `j_first`/`N_sys`
    select a shard of the 5*N_matrix perturbations per level; the first N_matrix (global) sit on the norm boundary.

    The interior perturbations are REJECTION samples of the norm ball, as upstream (utils.py:803-823); K6 gives up after
    256 draws and projects the last one onto the boundary, which changes the distribution. The acceptance rate of a
    uniform cube draw is ~0.31 for 2 x 2 (the shipped system: never exhausted) but ~6e-3 for 3 x 3 and ~4e-6 for
    4 x 4 in the Frobenius norm, where upstream's own loop would effectively not terminate either. The projected count
    is therefore always fetched and a non-zero count raises unless allow_projected=True."""
    total = 5 * N_matrix
    N_sys = total - j_first if N_sys is None else N_sys
    dA, sa = engine.sample_error_grid(seed, 0, n, n, N_sys, error_vec, N_matrix, norm_type, j_first=j_first,
                                      want_stats=True)
    dB, sb = engine.sample_error_grid(seed, 1, n, m, N_sys, error_vec, N_matrix, norm_type, j_first=j_first,
                                      want_stats=True)
    stats = {"rejected": sa["rejected"] + sb["rejected"], "projected": sa["projected"] + sb["projected"]}
    if stats["projected"] and not allow_projected:
        from .engine import EngineError
        raise EngineError("device_error_grids: %d interior perturbations exhausted the 256 rejection draws and were "
                          "projected onto the norm boundary (distribution changed); pass allow_projected=True to "
                          "accept that" % stats["projected"])
    return (dA, dB, stats) if return_stats else (dA, dB)


def perturbation_at(engine, seed, n, m, error_vec, N_matrix, norm_type, j, level):
    """(dA (n, n), dB (n, m)) of global perturbation j at error level `level` of the grids `device_error_grids`
    draws with the same arguments: K6 is counter-based, so drawing the single perturbation j (j_first=j, N_sys=1)
    gives exactly the entries the full grid holds there. This maps an index reported by
    `error_horizon_sweep(..., worst=True)` back to its sample."""
    if not 0 <= j < 5 * N_matrix or not 0 <= level < len(error_vec):
        raise ValueError("perturbation_at: j must be in [0, 5*N_matrix) and level in [0, len(error_vec))")
    dA = engine.sample_error_grid(seed, 0, n, n, 1, error_vec, N_matrix, norm_type, j_first=int(j))
    dB = engine.sample_error_grid(seed, 1, n, m, 1, error_vec, N_matrix, norm_type, j_first=int(j))
    return (dA[:, level].cpu().numpy().reshape(n, n), dB[:, level].cpu().numpy().reshape(n, m))


def grids_to_soa(error_A, error_B, level=None):
    """(n,n,N_sys,n_err), (n,m,N_sys,n_err) -> engine SoA [n*n][S], [n*m][S].
    level=None: every (system j, level i) pair, S = N_sys*n_err with s = j*n_err + i (the file's own C order);
    level=i: the N_sys systems of one level."""
    n, _, N_sys, n_err = error_A.shape
    m = error_B.shape[1]
    if level is None:
        return (np.ascontiguousarray(error_A.reshape(n * n, N_sys * n_err)),
                np.ascontiguousarray(error_B.reshape(n * m, N_sys * n_err)))
    return (np.ascontiguousarray(error_A[:, :, :, level].reshape(n * n, N_sys)),
            np.ascontiguousarray(error_B[:, :, :, level].reshape(n * m, N_sys)))


def synth_problem(n=4, m=2, seed=0, rho_target=1.05):
    """cfg-synth (SURVEY 8d.4/5): A_true = G * rho_target / rho(G), G ~ N(0,1)^{n x n}; B_true ~ N(0,1)^{n x m};
    Q = I, R = I, P = Q; re-drawn until (A, B) is controllable with a well-conditioned Gramian."""
    rng = np.random.default_rng(seed)
    while True:
        G = rng.normal(size=(n, n))
        A = G * (rho_target / np.max(np.abs(np.linalg.eigvals(G))))
        B = rng.normal(size=(n, m))
        C = np.hstack([np.linalg.matrix_power(A, k) @ B for k in range(n)])
        if np.linalg.matrix_rank(C) == n and np.linalg.cond(C @ C.T) < 1e12:
            return A, B, np.eye(n), np.eye(m)


def synth_samples_soa(n, m, S, seed=1, first=0, e=0.01, block=1 << 16, out=None, aos=False):
    """Seeded, shard-invariant synthetic samples in the engine's SoA layout: dA [n*n][S], dB [n*m][S] ~ U[-e, e],
    x0 [n][S] ~ N(0, I). Block b (of `block` samples) comes from Philox(key=[seed, stream], counter=[0,0,0,b]), so a
    rank asking for global samples [first, first+S) gets exactly what a single-GPU run would see there.
    `out` = (dA, dB, x0) preallocated arrays (e.g. views of pinned tensors).
    aos=True writes the array-of-matrices layout of the large-n path (K4) instead: dA [S][n*n], dB [S][n*m], x0 [S][n]
    (the same stream, transposed)."""
    if out is None:
        out = (np.empty((S, n * n)), np.empty((S, n * m)), np.empty((S, n))) if aos else \
            (np.empty((n * n, S)), np.empty((n * m, S)), np.empty((n, S)))
    dA, dB, x0 = out
    b0, b1 = first // block, (first + S - 1) // block
    pos = 0
    for b in range(b0, b1 + 1):
        g = np.random.Generator(np.random.Philox(key=[seed, _PHILOX_STREAM], counter=[0, 0, 0, b]))
        a = g.uniform(-e, e, size=(block, n * n))
        bb = g.uniform(-e, e, size=(block, n * m))
        xx = g.standard_normal(size=(block, n))
        lo = max(first, b * block) - b * block
        hi = min(first + S, (b + 1) * block) - b * block
        cnt = hi - lo
        if aos:
            dA[pos:pos + cnt] = a[lo:hi]
            dB[pos:pos + cnt] = bb[lo:hi]
            x0[pos:pos + cnt] = xx[lo:hi]
        else:
            dA[:, pos:pos + cnt] = a[lo:hi].T
            dB[:, pos:pos + cnt] = bb[lo:hi].T
            x0[:, pos:pos + cnt] = xx[lo:hi].T
        pos += cnt
    return dA, dB, x0
