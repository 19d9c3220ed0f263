"""Development A/B (GPU box): K1's closed-loop cost from the characteristic polynomial (default) against the Lyapunov
doubling for every sample (LQMPC_K1_LYAP=doubling), both in one process and alternating, at bench.py's headline size
(cfg-synth-4-2-10: n = 4, m = 2, N = 10, 1.25e7 samples, e = 0.01, same seeds). Prints one JSON line: CUDA-event time
per launch (mean, spread, every round) per path, the largest relative J and ratio difference between the paths, and
the card's name and power limit. Not part of the product."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from lq_mpc_b200 import sampling as sp  # noqa: E402
from lq_mpc_b200.engine import Engine  # noqa: E402

MODES = {"poly": None, "doubling": "doubling"}


def set_mode(mode):
    if MODES[mode] is None:
        os.environ.pop("LQMPC_K1_LYAP", None)
    else:
        os.environ["LQMPC_K1_LYAP"] = MODES[mode]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": pl}
    except Exception as e:  # noqa: BLE001 - the timing is still worth printing
        return {"error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=12_500_000)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--launches", type=int, default=20, help="timed launches per path and round")
    args = ap.parse_args()
    n, m, N, S = 4, 2, 10, args.samples
    eng = Engine(0)
    A, B, Q, R = sp.synth_problem(n, m, seed=0)
    eng.set_problem(A, B, Q, R, Q, None, None, 30)
    hA = np.empty((n * n, S)); hB = np.empty((n * m, S)); hx = np.empty((n, S))
    sp.synth_samples_soa(n, m, S, seed=1, first=0, e=0.01, out=(hA, hB, hx))
    dA, dB, x0 = (torch.from_numpy(a).cuda() for a in (hA, hB, hx))
    res = {}
    for mode in MODES:
        set_mode(mode)
        r = eng.eval_batch(dA, dB, x0, N, N)
        res[mode] = {k: r[k].cpu().numpy().copy() for k in ("J", "rho", "ratio", "flags")}
    diff = {k: float(np.max(np.abs(res["poly"][k] - res["doubling"][k]) / np.abs(res["doubling"][k])))
            for k in ("J", "ratio")}
    same = {k: bool(np.array_equal(res["poly"][k], res["doubling"][k])) for k in ("rho", "flags")}
    times = {mode: [] for mode in MODES}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for mode in MODES:
            set_mode(mode)
            for _ in range(3):
                eng.eval_batch(dA, dB, x0, N, N)
            e0.record()
            for _ in range(args.launches):
                eng.eval_batch(dA, dB, x0, N, N)
            e1.record()
            torch.cuda.synchronize()
            times[mode].append(e0.elapsed_time(e1) / args.launches)
    set_mode("poly")
    out = {"workload": "cfg-synth-4-2-10 K1 alone", "samples": S, "card": card(),
           "ms_per_launch": {k: {"mean": float(np.mean(v)), "min": float(np.min(v)), "max": float(np.max(v)),
                                 "rounds": v} for k, v in times.items()},
           "speedup": float(np.mean(times["doubling"]) / np.mean(times["poly"])),
           "max_rel_diff": diff, "bit_equal": same}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
