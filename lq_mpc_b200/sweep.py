"""Batch sweep driver for error magnitude x horizon (BASELINE.json configs[2]; SURVEY 8d.3).

The reference's `LQ_RDP_Behavior_Multiple.data_generation` (utils_class.py:766-959) fills two tables — error level at
the nominal horizon (802-859) and horizon at one hard-coded level (886-942) — with a Python triple loop, 100 systems
per column. `error_horizon_sweep` is the same body evaluated on the FULL grid (every error level x every horizon) at
10^5 perturbations per level: for one horizon N, every (perturbation j, level i) pair is one sample of a single batch
(s = j*n_err + i, the reference file's own C order) and the five quantities come from three launches

    K2a  M_V   = max_k V_N(x0_k)  over the ring of initial states        (utils_class.py:813-824)
    K2b  J_T   closed loop on the true plant, exact input-box QP per step (utils_class.py:828-833)
    K3   alpha, beta, xi, eta, J_bound (DARE gain computed in-kernel)     (utils_class.py:840-859)

followed by K5 on the [quantity][level] columns; only the per-column statistics (what the reference's plotters
draw, utils.py:895-898) leave the GPU. Multi-GPU: perturbations are sharded contiguously; the column moments are
merged by the one all-gather of `stats.column_stats`.

1 eval = one (perturbation, level, horizon) triple = 8 open-loop QPs + T closed-loop QPs + 1 DARE + the bound.
"""
from __future__ import annotations

import time
from typing import Optional, Sequence

import numpy as np

from . import stats as _stats
from .sampling import grids_to_soa
from .utils import circle_generator, local_radius

QUANTITIES = ("true_cost", "bound", "alpha", "beta", "xi", "eta", "M_V")


def _strided_columns(v, n_err):
    """[S = N_sys*n_err] device vector (s = j*n_err + i) -> contiguous [n_err][N_sys] table (one column per level)."""
    return v.reshape(-1, n_err).t().contiguous()


def error_horizon_sweep(engine, error_A, error_B, error_vec: Sequence[float], horizons: Sequence[int], F_u, Q,
                        N_points: int = 8, ext_radius_max: float = 1.5, p=(0.1, 1.0, 0.6), T: int = 30,
                        strict_reference: bool = True, group=None, keep_tables: bool = False,
                        shard: Optional[tuple] = None, phase_times: bool = False, fused_horizons: bool = False,
                        quantiles: Optional[Sequence[float]] = None, worst: bool = False,
                        j_first: Optional[int] = None, infinite_horizon: bool = False, T_max: int = 1000):
    """Full error-level x horizon sweep on an engine whose TRUE problem (A, B, Q, R, box, N_opc) is already set.

    error_A (n,n,N_sys,n_err), error_B (n,m,N_sys,n_err): the reference's grid layout (numpy) — `shard` = (rank, world)
    then restricts this process to its contiguous slice of the N_sys axis — or the SoA device tensors of
    `sampling.device_error_grids` (this rank's shard, generated in HBM by K6). Returns a dict:
      'error', 'horizon', 'V_expert', 'x_start', 'epsilon_lqr',
      '<q>_<stat>' for q in QUANTITIES, stat in max/min/mean/std : arrays [n_err][n_horizons],
      'ratio_true_max' / 'ratio_bound_max' (performance ratios J / V_expert, worst case per cell),
      'n_invalid' [n_err][n_horizons] (samples whose bound is void or raised in the reference),
      'n_failed' [n_err][n_horizons] (samples with an incomplete solve: QP_MAXITER / *_NOCONV / CHOL_FAIL — expected 0),
      'evals', 'seconds' (device time of the sweep loop), and with keep_tables the raw [n_horizons][q][n_err][N_sys];
      with phase_times 'phase_seconds' = device time per kernel family over the whole sweep (CUDA events between the
      launches, read after the loop: no synchronisation is added).

    fused_horizons=True evaluates the horizon axis with the range entry points: ONE mpc_solve_range over
    min(horizons)..max(horizons) (one Riccati sweep per sample serves every horizon; the requested horizons are picked
    from its [H] slots), the closed loops per horizon as before, and ONE bounds_range with the [H][S] M_V. Same keys,
    same phase names; M_V and true_cost bit-equal to the default mode, the bound statistics within 1e-9 relative
    (the Gram-spectrum search of the range stops at the same tolerance along a different path).

    Order statistics (opt-in; without them the sweep issues the same launches and returns the same values):
      quantiles=(0.05, 0.5, 0.95) adds '<q>_quantile' [len(quantiles)][n_err][n_horizons] for q in QUANTITIES, equal
        to np.quantile over the finite entries of each cell (see stats.column_quantiles), and 'quantiles'. The
        per-horizon tables stay on the device ([n_horizons][q][n_err][N_sys] doubles) and ONE radix selection over
        all their columns runs after the loop: one all-reduce per radix pass, whatever the number of horizons.
      worst=True adds '<q>_argmax' / '<q>_argmin' [n_err][n_horizons] int64: the global perturbation index j (the
        reference file's N_sys axis) attaining '<q>_max' / '<q>_min', lowest j on ties, -1 for a cell without a
        finite entry. j_first = the global index of this rank's first perturbation: by default the shard's start for
        numpy grids, 0 for device grids (pass the j_first given to `device_error_grids`). `sampling.perturbation_at`
        regenerates the perturbation of a K6 grid from its index.

    infinite_horizon=True (opt-in like the order statistics) adds, in both modes, one simulate_inf_batch per horizon
    (same grids and x_start; T_max bounds the steps before the certificate, see Engine.simulate_inf_batch) and the
    reduced quantity 'true_cost_inf' (the certified J_inf = lim J_T) with the statistics of every other quantity
    (moments, and '_quantile' / '_argmax' / '_argmin' when those are on), 'ratio_true_inf_max', and the counts
    'n_uncertified' / 'n_inf' [n_err][n_horizons] of its NaN (not certified within T_max) and +inf (unstable) entries,
    which the statistics leave out. Its launches are timed with the closed loops ('simulate' phase). Only J_inf is
    read from them: an incomplete solve in their steps before the certificate is not added to 'n_failed', which keeps
    every key of the plain sweep as it is without the option.
    """
    import torch
    n_err = len(error_vec)
    quants = QUANTITIES + ("true_cost_inf",) if infinite_horizon else QUANTITIES
    on_device = isinstance(error_A, torch.Tensor)          # SoA [n*n][N_sys*n_err] from K6 (already this rank's shard)
    if on_device:
        n = engine.n
        N_sys = error_A.shape[1] // n_err
    else:
        n = error_A.shape[0]
        N_sys_all = error_A.shape[2]
        if shard is not None:
            lo, hi = _stats.shard_bounds(N_sys_all, shard[0], shard[1])
            error_A, error_B = error_A[:, :, lo:hi, :], error_B[:, :, lo:hi, :]
        N_sys = error_A.shape[2]
        if j_first is None and shard is not None:
            j_first = lo
    if j_first is None:
        j_first = 0
    # ---- nominal quantities (utils_class.py:757-764, 782-786)
    K_lqr = engine.dlqr_batch(S=1)["K"].cpu().numpy()[:, 0].reshape(-1, n)
    eps_lqr = local_radius(F_u, -K_lqr, Q)
    x0_vec = circle_generator(N_points, ext_radius_max, eps_lqr, Q)
    x_start = x0_vec[:, 1].copy()
    V_expert = float(engine.mpc_solve_batch(None, None, engine.N_opc, pts=x_start[None], S=1)["V"][0, 0])
    if on_device:
        dA, dB = error_A, error_B
    else:
        dA, dB = grids_to_soa(np.ascontiguousarray(error_A), np.ascontiguousarray(error_B))
        dA, dB = engine._dev(dA), engine._dev(dB)
    e_per = engine._dev(np.tile(np.asarray(error_vec, dtype=np.float64), N_sys))
    ring = engine._dev(x0_vec.T.copy())
    x_start_d = engine._dev(x_start)                               # staged once: the loop below issues no H2D copy
    res = {q + "_" + s: np.zeros((n_err, len(horizons))) for q in quants for s in ("max", "min", "mean", "std")}
    n_invalid = np.zeros((n_err, len(horizons)))
    n_failed = np.zeros((n_err, len(horizons)))
    n_uncertified = np.zeros((n_err, len(horizons)))
    n_inf = np.zeros((n_err, len(horizons)))
    tables = [] if keep_tables else None
    dev_moments, dev_counts, dev_argext = [], [], []
    qs = _stats.check_quantiles(quantiles) if quantiles is not None else None
    if qs is not None:                     # every horizon's table, kept for the one selection after the loop
        qtab = torch.empty((len(horizons), len(quants) * n_err, N_sys), dtype=torch.float64, device=engine.device)
    torch.cuda.synchronize(engine.device)
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    marks = []

    def mark():
        if phase_times:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            marks.append(ev)

    def reduce_horizon(h, rs_flags, mv, sim, b, sinf=None):
        parts = [_strided_columns(v, n_err) for v in
                 (sim["J_T"], b["bound"], b["alpha"], b["beta"], b["xi"], b["eta"], mv)]
        if sinf is not None:
            parts.append(_strided_columns(sinf["J_inf"], n_err))
        cols = torch.cat(parts, dim=0) if qs is None else torch.cat(parts, dim=0, out=qtab[h])
        if worst:
            dev_argext.append(_stats.pack_argext(*engine.column_argext_raw(cols, j_first)))
        # K5 + the all-gather stay on the stream; the moments are read back ONCE after the loop (a .cpu() here would
        # drain the launch queue every horizon: ~0.4 ms of idle GPU per horizon, 5 % of the round-2 sweep)
        dev_moments.append(_stats.column_moments_device(engine, cols, group))
        bad = ((b["flags"] & (32 | 512)) != 0).to(torch.float64)       # BOUND_INVALID | DOMAIN_ERROR
        # incomplete solves (QP_MAXITER | DARE_NOCONV | LYAP_NOCONV | EIG_NOCONV | CHOL_FAIL) anywhere in the cell
        any_f = b["flags"] | sim["flags"]
        for row in rs_flags:
            any_f = any_f | row
        fail = ((any_f & (4 | 8 | 64 | 128 | 256)) != 0).to(torch.float64)
        counts = [bad, fail]
        if sinf is not None:
            counts += [torch.isnan(sinf["J_inf"]).to(torch.float64), torch.isinf(sinf["J_inf"]).to(torch.float64)]
        dev_counts.append(torch.stack([_strided_columns(c, n_err).sum(dim=1) for c in counts]))
        if keep_tables:
            tables.append(cols.reshape(len(quants), n_err, N_sys).cpu().numpy())

    if not fused_horizons:
        for h, N in enumerate(horizons):
            N = int(N)
            mark()
            rs = engine.mpc_solve_batch(dA, dB, N, pts=ring, want=("M_V", "flags"))
            mv = rs["M_V"]
            mark()
            sim = engine.simulate_batch(dA, dB, N, T, x0_shared=x_start_d, want=("J_T", "flags"))
            sinf = engine.simulate_inf_batch(dA, dB, N, T_max, x0_shared=x_start_d, want=("J_inf",)) \
                if infinite_horizon else None
            mark()
            b = engine.bounds_batch(dA, dB, N, e_per, e_per, mv, x_start_d, p, V_expert,
                                    strict_reference=strict_reference)
            mark()
            reduce_horizon(h, rs["flags"], mv, sim, b, sinf)
    else:
        N_lo, N_hi = int(min(horizons)), int(max(horizons))
        pick = [int(N) - N_lo for N in horizons]                      # slots of the covering range
        mark()
        rs = engine.mpc_solve_range(dA, dB, N_lo, N_hi, pts=ring, want=("M_V", "flags"))
        mark()
        sims = [engine.simulate_batch(dA, dB, int(N), T, x0_shared=x_start_d, want=("J_T", "flags")) for N in horizons]
        sinfs = [engine.simulate_inf_batch(dA, dB, int(N), T_max, x0_shared=x_start_d, want=("J_inf",))
                 for N in horizons] if infinite_horizon else [None] * len(horizons)
        mark()
        br = engine.bounds_range(dA, dB, N_lo, N_hi, e_per, e_per, rs["M_V"], x_start_d, p, V_expert,
                                 strict_reference=strict_reference, detail=False)
        mark()
        for h, N in enumerate(horizons):
            k = pick[h]
            b = {q: br[q][k] for q in ("alpha", "beta", "xi", "eta", "bound", "flags")}
            reduce_horizon(h, rs["flags"][k], rs["M_V"][k], sims[h], b, sinfs[h])
    if qs is not None:
        keys = _stats.column_quantile_keys(engine, qtab.view(-1, N_sys), qs,
                                           torch.stack(dev_moments)[:, :, :, 2].sum(dim=1).reshape(-1), group)
    if worst:
        argext = _stats.gather_rows(torch.stack(dev_argext), group)  # [ranks][n_horizons][cols][4]
    host_moments = torch.stack(dev_moments).cpu().numpy()              # [n_horizons][ranks][cols][6]
    host_counts = torch.stack(dev_counts).cpu().numpy()                # [n_horizons][2][n_err]
    if qs is not None:
        host_keys = keys.cpu().numpy()
    if worst:
        host_argext = argext.cpu().numpy()
    mark()
    e1.record()
    torch.cuda.synchronize(engine.device)
    for h in range(len(horizons)):
        st = _stats.merge_moments(host_moments[h])                     # [len(quants)*n_err] columns
        for qi, q in enumerate(quants):
            for sname in ("max", "min", "mean", "std"):
                res[q + "_" + sname][:, h] = st[sname][qi * n_err:(qi + 1) * n_err]
        n_invalid[:, h] = host_counts[h, 0]
        n_failed[:, h] = host_counts[h, 1]
        if infinite_horizon:
            n_uncertified[:, h] = host_counts[h, 2]
            n_inf[:, h] = host_counts[h, 3]
    phases = None
    if phase_times:
        phases = {"ring_solves": 0.0, "simulate": 0.0, "bounds": 0.0, "stats_and_packing": 0.0}
        names = list(phases)
        for i in range(len(marks) - 1):
            phases[names[i % 4]] += marks[i].elapsed_time(marks[i + 1]) * 1e-3
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        counts = [n_invalid, n_failed] + ([n_uncertified, n_inf] if infinite_horizon else [])
        t = torch.from_numpy(np.stack(counts)).to(engine.device)   # (column_stats merged the moments)
        dist.all_reduce(t, group=group)
        t = t.cpu().numpy()
        n_invalid, n_failed = t[0], t[1]
        if infinite_horizon:
            n_uncertified, n_inf = t[2], t[3]
    res.update({"error": np.asarray(error_vec, dtype=np.float64), "horizon": np.asarray(horizons),
                "V_expert": V_expert, "x_start": x_start, "epsilon_lqr": eps_lqr, "n_invalid": n_invalid, "n_failed": n_failed,
                "ratio_true_max": res["true_cost_max"] / V_expert, "ratio_bound_max": res["bound_max"] / V_expert,
                "evals": int(N_sys) * n_err * len(horizons), "seconds": e0.elapsed_time(e1) * 1e-3,
                "wall_seconds": time.perf_counter() - t0})
    if infinite_horizon:
        res.update({"ratio_true_inf_max": res["true_cost_inf_max"] / V_expert, "n_uncertified": n_uncertified,
                    "n_inf": n_inf})
    n_q = len(quants)
    if qs is not None:
        qv = _stats.finish_quantiles(host_keys, host_moments[:, :, :, 2].sum(axis=1).reshape(-1), qs)
        qv = qv.reshape(len(qs), len(horizons), n_q, n_err)
        for qi, q in enumerate(quants):
            res[q + "_quantile"] = np.ascontiguousarray(qv[:, :, qi, :].transpose(0, 2, 1))
        res["quantiles"] = qs
    if worst:
        ax = _stats.merge_argext(host_argext.reshape(host_argext.shape[0], -1, 4))
        for name in ("argmax", "argmin"):
            a = ax[name].reshape(len(horizons), n_q, n_err)
            for qi, q in enumerate(quants):
                res[q + "_" + name] = np.ascontiguousarray(a[:, qi, :].T)
    if keep_tables:
        res["tables"] = np.stack(tables)
    if phases is not None:
        res["phase_seconds"] = phases
    return res
