#!/usr/bin/env python
"""K2b's finite closed loop (simulate_batch, T = 30) against K2c's certified infinite-horizon cost
(simulate_inf_batch, T_max = 1000) on the cfg-sweep-f grids, in one process.

Inputs as bench.py's measure_sweep builds them: the 2-state example with the input box, 10 error levels x 10^5
perturbations from K6 (seed 20240522, Frobenius norm), the shared initial state x_start of the sweep, horizons N = 7
and 50. Both calls are warmed up; then each rep times one window of --calls back-to-back calls per side with CUDA
events, the sides alternating, --reps times. Prints one JSON line: per horizon the per-call milliseconds of every
window and their median for both calls, the histogram of the certified step tau, the counts of
uncertified / unstable samples, the largest |J_inf - J_T(30)| / J_T(30), and the card's name and power limit read in
the same run."""
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--per-level", type=int, default=100_000)
    ap.add_argument("--horizons", type=int, nargs="+", default=[7, 50])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--calls", type=int, default=200, help="calls per timed window")
    ap.add_argument("--T", type=int, default=30)
    ap.add_argument("--T-max", type=int, default=1000)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    import torch
    from lq_mpc_b200 import sampling as sp
    from lq_mpc_b200.engine import Engine
    from oracle.np_oracle import circle_generator, dlqr, local_radius
    if not torch.cuda.is_available():
        raise SystemExit("simulate_inf_bench: needs a CUDA device")
    A = np.array([[1, 0.7], [0.12, 0.4]]); B = np.array([[1], [1.2]])
    Q, R, lo, hi = 2 * np.eye(2), np.eye(1), np.array([-0.1]), np.array([0.1])
    eng = Engine(0)
    eng.set_problem(A, B, Q, R, Q, lo, hi, 30)
    error_vec = np.linspace(1e-3, 1e-2, 10)
    eA, eB = sp.device_error_grids(eng, 2, 1, error_vec, a.per_level // 5, "f", seed=20240522, j_first=0,
                                   N_sys=a.per_level)
    x_start = circle_generator(8, 1.5, local_radius(lo, hi, -dlqr(A, B, Q, R)[0], Q), Q)[:, 1].copy()
    xs = eng._dev(x_start)
    S = eA.shape[1]
    calls = {"simulate_T%d" % a.T: lambda N: eng.simulate_batch(eA, eB, N, a.T, x0_shared=xs, want=("J_T", "flags")),
             "simulate_inf_Tmax%d" % a.T_max: lambda N: eng.simulate_inf_batch(eA, eB, N, a.T_max, x0_shared=xs)}
    out = {"workload": "cfg-sweep-f grids", "samples": S, "reps": a.reps, "calls_per_window": a.calls, "card": card(),
           "horizons": {}}
    for N in a.horizons:
        last = {k: f(N) for k, f in calls.items()}                  # warm-up, and the outputs compared below
        times = {k: [] for k in calls}
        for _ in range(a.reps):
            for k, f in calls.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.calls):
                    f(N)
                e1.record()
                torch.cuda.synchronize()
                times[k].append(e0.elapsed_time(e1) / a.calls)
        JT = last["simulate_T%d" % a.T]["J_T"].cpu().numpy()
        inf = {k: v.cpu().numpy() for k, v in last["simulate_inf_Tmax%d" % a.T_max].items()}
        tau = inf["T_cert"]
        vals, counts = np.unique(tau, return_counts=True)
        ok = tau >= 0
        out["horizons"][str(N)] = {
            "ms_per_call_median": {k: float(np.median(v)) for k, v in times.items()},
            "ms_per_call": times,
            "tau_histogram": {str(int(v)): int(c) for v, c in zip(vals, counts)},
            "n_uncertified": int(np.sum(np.isnan(inf["J_inf"]))), "n_inf": int(np.sum(np.isinf(inf["J_inf"]))),
            "max_rel_J_inf_vs_J_T": float(np.max(np.abs(inf["J_inf"][ok] - JT[ok]) / JT[ok])) if ok.any() else None}
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
