"""Cost and effect of the worst ratio over every initial state on synth_problem(4, 2), N = 10 (DESIGN.md §4).

1. ratio_sup_batch value only and with the gradient, each against eval_grad_batch (the per-x0 gradient pass), on the
   same 10^6 samples, in alternating windows of CUDA-event-timed calls after a warm-up of every side.
2. worst_case_search_sup from the 10^4 samples of largest gamma for norm 'max' (synthetic samples U[-e, e]) and 'f'
   (K6 grids), e = 0.01 and 0.05: ms per call of the ascent, mean accepted steps, the share of runs ending on the
   budget, the sampled against the ascended maximum gamma, and worst_case_search's (per-x0) best ratio on the same
   samples for comparison.

The card name and power limit are read in the same run. Writes one JSON line to stdout and to --out when given.
Usage: python scripts/ratio_sup_bench.py [--samples 1000000] [--starts 10000] [--rounds 6] [--out FILE]"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from worst_case_bench import card, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=1_000_000)
    ap.add_argument("--starts", type=int, default=10_000)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from lq_mpc_b200.engine import FLAG_ASCENT_MAXITER, Engine
    from lq_mpc_b200.sampling import device_error_grids, synth_problem, synth_samples_soa
    from lq_mpc_b200.worst_case import worst_case_search, worst_case_search_sup
    if not torch.cuda.is_available():
        raise SystemExit("ratio_sup_bench.py needs a CUDA device")
    eng = Engine(0)
    A, B, Q, R = synth_problem(4, 2, seed=0)
    eng.set_problem(A, B, Q, R, Q, None, None, 30)
    N, S = 10, a.samples
    res = {"card": card(), "problem": "synth_problem(4, 2), N = 10", "samples": S}

    dA, dB, x0 = (eng._dev(v) for v in synth_samples_soa(4, 2, S, seed=1, e=0.01))
    sides = {"eval_grad_batch": lambda: eng.eval_grad_batch(dA, dB, x0, N),
             "ratio_sup_value": lambda: eng.ratio_sup_batch(dA, dB, N),
             "ratio_sup_grad": lambda: eng.ratio_sup_batch(dA, dB, N, grad=True)}
    for f in sides.values():
        f(); f()
    torch.cuda.synchronize()
    win = {k: [] for k in sides}
    for _ in range(a.rounds):
        for k, f in sides.items():
            win[k].append(timed(torch, f, a.calls))
    for k in sides:
        res[k + "_ms"] = float(np.median(win[k]))
    res["value_over_eval_grad"] = res["ratio_sup_value_ms"] / res["eval_grad_batch_ms"]
    res["grad_over_eval_grad"] = res["ratio_sup_grad_ms"] / res["eval_grad_batch_ms"]
    res["windows"] = {"rounds": a.rounds, "calls_per_window": a.calls, **{k + "_ms": v for k, v in win.items()}}
    g = eng.ratio_sup_batch(dA, dB, N)
    res["gap_median"] = float(g["gap"].median().item())
    del dA, dB, x0, g

    x_rng = np.random.default_rng(3)
    asc = []
    for norm in ("max", "f"):
        for e in (0.01, 0.05):
            if norm == "max":
                dA, dB, x0 = (eng._dev(v) for v in synth_samples_soa(4, 2, S, seed=2, e=e))
            else:
                dA, dB = device_error_grids(eng, 4, 2, [e], S // 5, "f", allow_projected=True)
                x0 = eng._dev(x_rng.normal(size=(4, dA.shape[1])))
            r = worst_case_search_sup(eng, dA, dB, N, e, e, norm, top_k=a.starts)
            per = worst_case_search(eng, dA, dB, x0, N, e, e, norm, top_k=a.starts)
            idx = r["start_index"]
            sA, sB = dA[:, idx].contiguous(), dB[:, idx].contiguous()
            call = lambda: eng.worst_case_sup_batch(sA, sB, N, e, e, norm)
            call()
            torch.cuda.synchronize()
            ms = [timed(torch, call, 3) for _ in range(3)]
            fl = r["flags"]
            k = int(idx.numel())
            asc.append({"norm": norm, "e": e, "samples": int(dA.shape[1]), "starts": k,
                        "ms_per_call": float(np.median(ms)),
                        "mean_accepted_steps": float(r["iters"].double().mean().item()),
                        "sampled_max_gamma": r["sampled_max_ratio"], "ascended_max_gamma": r["best_ratio"],
                        "excess_gamma": (r["best_ratio"] - 1) / (r["sampled_max_ratio"] - 1)
                        if r["n_unstable"] == 0 else None,
                        "n_unstable": r["n_unstable"],
                        "maxiter_share": int(((fl & FLAG_ASCENT_MAXITER) != 0).sum().item()) / max(k, 1),
                        "n_converged": int((fl == 0).sum().item()),
                        "per_x0_sampled_max_ratio": per["sampled_max_ratio"],
                        "per_x0_ascended_max_ratio": per["best_ratio"], "per_x0_n_unstable": per["n_unstable"]})
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
