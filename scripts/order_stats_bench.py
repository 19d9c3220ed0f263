#!/usr/bin/env python
"""Cost of the exact column quantiles and arg-extremes (K5 radix selection / argext), in one process.

Part 1, the kernels on three table shapes (random normal doubles generated on the device):
  sweep_horizon  70 columns x 10^5      (one horizon of cfg-sweep-f: 56 MB, fits the 126 MB L2)
  sweep_all      3 500 columns x 10^5   (all 50 horizons at once: 2.8 GB)
  synth          30 columns x 1.25e7    (cfg-synth's J / rho / ratio over 10 horizons: 3.0 GB)
Each is warmed up, then the selection of the quantiles (0.05, 0.5, 0.95) (8 x histogram + select) and one argext pass
are timed with CUDA events over --reps calls. Reported: ms per call, and bytes read per pass over the time of a pass,
as a fraction of the 7.7 TB/s HBM data-sheet figure (for the L2-resident shape this is not an HBM rate).
Part 2, cfg-sweep-f as bench.py builds it, with and without quantiles=(0.05, 0.5, 0.95), worst=True, alternating,
--sweep-reps timed sweeps each after a warm-up of both. Prints one JSON line with the card name and power limit."""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from scripts.sweep_fused_bench import card  # noqa: E402

HBM_TBPS = 7.7
QS = (0.05, 0.5, 0.95)
SHAPES = {"sweep_horizon": (70, 100_000), "sweep_all": (3_500, 100_000), "synth": (30, 12_500_000)}


def time_kernels(eng, cols, S, reps):
    import torch
    from lq_mpc_b200 import stats
    t = torch.randn((cols, S), dtype=torch.float64, device="cuda")
    counts = eng.column_moments_raw(t)[:, 2]
    qs = stats.check_quantiles(QS)

    def select():
        return stats.column_quantile_keys(eng, t, qs, counts)

    def argext():
        return eng.column_argext_raw(t, 0)
    out = {"cols": cols, "S": S, "table_bytes": cols * S * 8, "l2_resident": cols * S * 8 < 126e6}
    for name, fn, passes in (("quantiles", select, 8), ("argext", argext, 1)):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        rate = passes * cols * S * 8 / (ms * 1e-3) / 1e12
        out[name] = {"ms_per_call": ms, "passes": passes, "TBps_per_pass": rate, "hbm_fraction": rate / HBM_TBPS}
    keys = select().cpu().numpy()                          # spot check against numpy on the first column
    ref = np.quantile(t[0].cpu().numpy(), QS)
    got = stats.finish_quantiles(keys[:1], counts[:1].cpu().numpy(), qs)[:, 0]
    out["first_column_equals_numpy"] = bool(np.array_equal(got, ref))
    del t
    torch.cuda.empty_cache()
    return out


def time_sweep(eng, per_level, reps):
    import torch
    from lq_mpc_b200 import sampling as sp
    from lq_mpc_b200.sweep import error_horizon_sweep
    A = np.array([[1, 0.7], [0.12, 0.4]]); B = np.array([[1], [1.2]])
    Q, R, F_u = 2 * np.eye(2), np.eye(1), np.array([[10.0], [-10.0]])
    eng.set_problem(A, B, Q, R, Q, [-0.1], [0.1], 30)
    error_vec = np.linspace(1e-3, 1e-2, 10)
    horizons = list(range(1, 51))
    eA, eB = sp.device_error_grids(eng, 2, 1, error_vec, per_level // 5, "f", seed=20240522, j_first=0,
                                   N_sys=per_level)
    modes = {"plain": {}, "order_stats": {"quantiles": QS, "worst": True}}
    for kw in modes.values():
        error_horizon_sweep(eng, eA, eB, error_vec, horizons, F_u, Q, **kw)
    runs = {k: [] for k in modes}
    last = {}
    for _ in range(reps):
        for k, kw in modes.items():
            r = error_horizon_sweep(eng, eA, eB, error_vec, horizons, F_u, Q, phase_times=True, **kw)
            runs[k].append(r["seconds"])
            last[k] = r
    same = all(np.array_equal(np.asarray(last["plain"][k]), np.asarray(last["order_stats"][k]))
               for k in last["plain"] if k not in ("seconds", "wall_seconds", "phase_seconds"))
    out = {k: {"seconds_mean": float(np.mean(v)), "seconds": v} for k, v in runs.items()}
    out["added_seconds"] = out["order_stats"]["seconds_mean"] - out["plain"]["seconds_mean"]
    out["plain_keys_bit_equal"] = bool(same)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sweep-reps", type=int, default=3)
    ap.add_argument("--per-level", type=int, default=100_000)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("order_stats_bench: needs a CUDA device")
    from lq_mpc_b200.engine import Engine
    eng = Engine(0)
    out = {"card": card(), "quantiles": QS, "kernels": {}}
    for name in [s for s in a.shapes.split(",") if s]:
        out["kernels"][name] = time_kernels(eng, *SHAPES[name], a.reps)
    if a.sweep_reps > 0:
        out["sweep"] = time_sweep(eng, a.per_level, a.sweep_reps)
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
