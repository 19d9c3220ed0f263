#!/usr/bin/env python
"""cfg-sweep-f with and without the fused horizon axis (error_horizon_sweep(fused_horizons=...)), in one process.

Inputs exactly as bench.py's measure_sweep builds them: the 2-state example with the input box, 10 error levels,
horizons 1..50, 10^5 perturbations per level from K6 (seed 20240522, Frobenius norm). Both modes are warmed up on the
full grid, then timed --reps times each, alternating (default, fused, default, ...), with phase_times. Prints one JSON
line: the mean and per-rep seconds and phase seconds of both modes, the max relative difference of every statistic
between the modes (from the last sweep of each), and the card's name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        name, limit = [v.strip() for v in r.stdout.strip().split(",")]
        return {"name": name, "power_limit": limit}
    except Exception as exc:                                        # the run itself needs no nvidia-smi
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": "not read (%s)" % type(exc).__name__}


def max_rel_diff(a, b):
    fin = np.isfinite(b) & np.isfinite(a)
    mask_diff = int(np.sum(np.isfinite(a) != np.isfinite(b)))
    if not fin.any():
        return 0.0, mask_diff
    return float(np.max(np.abs(a[fin] - b[fin]) / np.maximum(np.abs(b[fin]), 1e-300))), mask_diff


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--per-level", type=int, default=100_000)
    ap.add_argument("--nmax", type=int, default=50)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    import torch
    from lq_mpc_b200 import sampling as sp
    from lq_mpc_b200.engine import Engine
    from lq_mpc_b200.sweep import QUANTITIES, error_horizon_sweep
    if not torch.cuda.is_available():
        raise SystemExit("sweep_fused_bench: needs a CUDA device")
    A = np.array([[1, 0.7], [0.12, 0.4]]); B = np.array([[1], [1.2]])
    Q, R, F_u = 2 * np.eye(2), np.eye(1), np.array([[10.0], [-10.0]])
    eng = Engine(0)
    eng.set_problem(A, B, Q, R, Q, [-0.1], [0.1], 30)
    error_vec = np.linspace(1e-3, 1e-2, 10)
    horizons = list(range(1, a.nmax + 1))
    eA, eB = sp.device_error_grids(eng, 2, 1, error_vec, a.per_level // 5, "f", seed=20240522, j_first=0,
                                   N_sys=a.per_level)
    torch.cuda.synchronize()
    modes = {"default": False, "fused": True}
    for fused in modes.values():                                   # warm-up: every shape of the timed sweeps
        error_horizon_sweep(eng, eA, eB, error_vec, horizons, F_u, Q, fused_horizons=fused)
    runs = {k: [] for k in modes}
    last = {}
    for _ in range(a.reps):
        for k, fused in modes.items():
            r = error_horizon_sweep(eng, eA, eB, error_vec, horizons, F_u, Q, phase_times=True, fused_horizons=fused)
            runs[k].append({"seconds": r["seconds"], "phase_seconds": r["phase_seconds"]})
            last[k] = r
    out = {"workload": "cfg-sweep-f", "per_level": a.per_level, "n_err": len(error_vec), "nmax": a.nmax,
           "evals": last["default"]["evals"], "reps": a.reps, "card": card()}
    for k in modes:
        ph = {p: float(np.mean([x["phase_seconds"][p] for x in runs[k]])) for p in runs[k][0]["phase_seconds"]}
        out[k] = {"seconds_mean": float(np.mean([x["seconds"] for x in runs[k]])),
                  "seconds": [x["seconds"] for x in runs[k]], "phase_seconds_mean": ph,
                  "phase_seconds": [x["phase_seconds"] for x in runs[k]]}
    out["speedup"] = out["default"]["seconds_mean"] / out["fused"]["seconds_mean"]
    diffs = {}
    for q in QUANTITIES:
        for st in ("max", "min", "mean", "std"):
            k = q + "_" + st
            rel, masks = max_rel_diff(last["fused"][k], last["default"][k])
            diffs[k] = rel if masks == 0 else {"max_rel": rel, "finite_mask_differences": masks}
    for k in ("n_invalid", "n_failed"):
        diffs[k + "_equal"] = bool(np.array_equal(last["fused"][k], last["default"][k]))
    out["max_rel_diff_fused_vs_default"] = diffs
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
