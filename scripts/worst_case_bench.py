"""Cost of the worst-case entry points on synth_problem(4, 2), N = 10 (DESIGN.md §4).

1. eval_batch (one horizon) against eval_grad_batch on the same 10^6 samples, in alternating windows of CUDA-event-timed
   calls after a warm-up of both.
2. worst_case_batch from the 10^4 samples of largest K1 ratio (worst_case_search's starts) for norm 'max' (synthetic
   samples U[-e, e]) and 'f' (K6 grids), e = 0.01 and 0.05: ms per call, mean accepted steps per start, and the sampled
   against the ascended maximum ratio.

The card name and power limit are read in the same run. Writes one JSON line to stdout and to --out when given.
Usage: python scripts/worst_case_bench.py [--samples 1000000] [--starts 10000] [--rounds 6] [--out FILE]"""
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
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from lq_mpc_b200.engine import FLAG_ASCENT_MAXITER, FLAG_UNSTABLE, Engine
    from lq_mpc_b200.sampling import device_error_grids, synth_problem, synth_samples_soa
    from lq_mpc_b200.worst_case import worst_case_search
    if not torch.cuda.is_available():
        raise SystemExit("worst_case_bench.py needs a CUDA device")
    eng = Engine(0)
    A, B, Q, R = synth_problem(4, 2, seed=0)
    eng.set_problem(A, B, Q, R, Q, None, None, 30)
    N, S = 10, a.samples
    res = {"card": card(), "problem": "synth_problem(4, 2), N = 10", "samples": S}

    dA, dB, x0 = (eng._dev(v) for v in synth_samples_soa(4, 2, S, seed=1, e=0.01))
    f1 = lambda: eng.eval_batch(dA, dB, x0, N, N)
    f2 = lambda: eng.eval_grad_batch(dA, dB, x0, N)
    for f in (f1, f2):
        f(); f()
    torch.cuda.synchronize()
    t1, t2 = [], []
    for _ in range(a.rounds):
        t1.append(timed(torch, f1, a.calls))
        t2.append(timed(torch, f2, a.calls))
    res["eval_batch_ms"] = float(np.median(t1))
    res["eval_grad_batch_ms"] = float(np.median(t2))
    res["grad_over_eval"] = res["eval_grad_batch_ms"] / res["eval_batch_ms"]
    res["windows"] = {"rounds": a.rounds, "calls_per_window": a.calls, "eval_ms": t1, "grad_ms": t2}
    del dA, dB, x0

    x_rng = np.random.default_rng(3)
    asc = []
    for norm in ("max", "f"):
        for e in (0.01, 0.05):
            if norm == "max":
                dA, dB, x0 = (eng._dev(v) for v in synth_samples_soa(4, 2, S, seed=2, e=e))
            else:
                dA, dB = device_error_grids(eng, 4, 2, [e], S // 5, "f", allow_projected=True)
                x0 = eng._dev(x_rng.normal(size=(4, dA.shape[1])))
            r = worst_case_search(eng, dA, dB, x0, N, e, e, norm, top_k=a.starts)
            idx = r["start_index"]
            sA, sB, sx = dA[:, idx].contiguous(), dB[:, idx].contiguous(), x0[:, idx].contiguous()
            call = lambda: eng.worst_case_batch(sA, sB, sx, N, e, e, norm)
            call()
            torch.cuda.synchronize()
            ms = [timed(torch, call, 3) for _ in range(3)]
            fl = r["flags"]
            asc.append({"norm": norm, "e": e, "starts": int(idx.numel()), "ms_per_call": float(np.median(ms)),
                        "mean_accepted_steps": float(r["iters"].double().mean().item()),
                        "sampled_max_ratio": r["sampled_max_ratio"], "ascended_max_ratio": r["best_ratio"],
                        "n_unstable": r["n_unstable"],
                        "n_maxiter": int(((fl & FLAG_ASCENT_MAXITER) != 0).sum().item()),
                        "n_converged": int((fl == 0).sum().item()),
                        "excess_ratio": (r["best_ratio"] - 1) / (r["sampled_max_ratio"] - 1)
                        if r["n_unstable"] == 0 else None})
            del dA, dB, x0
    res["ascent"] = asc
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    eng.close()


if __name__ == "__main__":
    main()
