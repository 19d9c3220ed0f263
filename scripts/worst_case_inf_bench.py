#!/usr/bin/env python
"""Cost and reach of the input-constrained worst-case entry points on the cfg-sweep-f grids (DESIGN.md §4).

Inputs as bench.py's measure_sweep builds them: the 2-state example with its input box, one error level (e = 1e-2) of
the K6 grids (seed 20240522, Frobenius norm), --samples perturbations, the sweep's shared initial state x_start.

1. For N = 7 and 50: simulate_inf_batch against simulate_inf_grad_batch on the same samples, both warmed up, then
   --rounds alternating windows of --calls CUDA-event-timed calls per side; median and spread of the per-call times.
2. For N = 7 and 50, on the entrywise box (samples U[-e, e]) and the Frobenius grids: worst_case_search_inf from the
   --starts samples of largest J_inf (ms per ascent call, mean accepted steps, the share ending with
   FLAG_ASCENT_MAXITER, sampled against ascended max J_inf, n_unstable), and worst_case_search on the same samples
   (the unconstrained law, x0 = x_start) for comparison, with K2c's J_inf at the unconstrained worst error.

The card name and power limit are read in the same run. Writes one JSON line to stdout and to --out when given."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except Exception as e:      # the number is still reported, marked without its power limit
        info["power_limit_and_max_sm_clock"] = "unavailable: %s" % e
    return info


def timed(torch, fn, calls):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / calls


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=1_000_000)
    ap.add_argument("--starts", type=int, default=10_000)
    ap.add_argument("--horizons", type=int, nargs="+", default=[7, 50])
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--e", type=float, default=1e-2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from lq_mpc_b200 import sampling as sp
    from lq_mpc_b200.engine import FLAG_ASCENT_MAXITER, Engine
    from lq_mpc_b200.worst_case import worst_case_search, worst_case_search_inf
    from oracle.np_oracle import circle_generator, dlqr, local_radius
    if not torch.cuda.is_available():
        raise SystemExit("worst_case_inf_bench.py needs a CUDA device")
    A = np.array([[1, 0.7], [0.12, 0.4]]); B = np.array([[1], [1.2]])
    Q, R, lo, hi = 2 * np.eye(2), np.eye(1), np.array([-0.1]), np.array([0.1])
    eng = Engine(0)
    eng.set_problem(A, B, Q, R, Q, lo, hi, 30)
    x_start = circle_generator(8, 1.5, local_radius(lo, hi, -dlqr(A, B, Q, R)[0], Q), Q)[:, 1].copy()
    xs = eng._dev(x_start)
    e = a.e
    gA, gB = sp.device_error_grids(eng, 2, 1, [e], a.samples // 5, "f", seed=20240522, j_first=0, N_sys=a.samples)
    bA, bB, _ = (eng._dev(v) for v in sp.synth_samples_soa(2, 1, gA.shape[1], seed=2, e=e))
    res = {"card": card(), "workload": "cfg-sweep-f grids, e = %g, shared x_start" % e, "samples": int(gA.shape[1]),
           "starts": a.starts, "horizons": {}}
    for N in a.horizons:
        f1 = lambda: eng.simulate_inf_batch(gA, gB, N, 1000, x0_shared=xs)
        f2 = lambda: eng.simulate_inf_grad_batch(gA, gB, N, 1000, x0_shared=xs)
        for f in (f1, f2):
            f(); f()
        torch.cuda.synchronize()
        t1, t2 = [], []
        for _ in range(a.rounds):
            t1.append(timed(torch, f1, a.calls))
            t2.append(timed(torch, f2, a.calls))
        h = {"simulate_inf_ms": float(np.median(t1)), "simulate_inf_grad_ms": float(np.median(t2)),
             "windows": {"rounds": a.rounds, "calls_per_window": a.calls, "simulate_inf_ms": t1,
                         "simulate_inf_grad_ms": t2}}
        h["grad_over_value"] = h["simulate_inf_grad_ms"] / h["simulate_inf_ms"]
        searches = []
        for norm, dA, dB in (("max", bA, bB), ("f", gA, gB)):
            r = worst_case_search_inf(eng, dA, dB, N, e, e, norm, x0_shared=xs, top_k=a.starts)
            idx = r["start_index"]
            sA, sB = dA[:, idx].contiguous(), dB[:, idx].contiguous()
            call = lambda: eng.worst_case_inf_batch(sA, sB, N, e, e, norm, x0_shared=xs)
            call()
            torch.cuda.synchronize()
            ms = [timed(torch, call, 3) for _ in range(3)]
            fl = r["flags"]
            u = worst_case_search(eng, dA, dB, xs, N, e, e, norm, top_k=a.starts)
            bu = int(torch.argmax(torch.nan_to_num(u["J"], nan=-float("inf"))).item())
            at_u = eng.simulate_inf_batch(u["dA"][:, bu:bu + 1], u["dB"][:, bu:bu + 1], N, 1000, x0_shared=xs)
            bc = int(torch.argmax(torch.nan_to_num(r["J"], nan=-float("inf"))).item())
            searches.append({
                "norm": norm, "ms_per_call": float(np.median(ms)), "ms_windows": ms,
                "mean_accepted_steps": float(r["iters"].double().mean().item()),
                "share_ascent_maxiter": float(((fl & FLAG_ASCENT_MAXITER) != 0).double().mean().item()),
                "sampled_max_J_inf": r["sampled_max_J"], "ascended_max_J_inf": r["best_J"],
                "n_unstable": r["n_unstable"], "n_uncertified": r["n_uncertified"],
                "unconstrained_ascended_max_J": float(u["J"][bu].item()),
                "J_inf_at_unconstrained_worst_error": float(at_u["J_inf"][0].item()),
                "best_error_distance_fro": float(torch.sqrt(torch.sum((r["dA"][:, bc] - u["dA"][:, bu]) ** 2) +
                                                            torch.sum((r["dB"][:, bc] - u["dB"][:, bu]) ** 2)).item())})
        h["search"] = searches
        res["horizons"][str(N)] = h
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    eng.close()


if __name__ == "__main__":
    main()
