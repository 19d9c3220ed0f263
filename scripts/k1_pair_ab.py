"""Development A/B (GPU box): K1 with two samples per thread (default) against one sample per thread
(LQMPC_K1_PAIR=0), both in one process and alternating, at bench.py's headline size (cfg-synth-4-2-10: n = 4, m = 2,
N = 10, 1.25e7 samples, e = 0.01, same seeds), through eval_batch and through the seeded entry point (operands drawn in
the kernel, column moments behind it). Prints one JSON line: CUDA-event time per launch (mean, spread, every round) per
path and entry point, whether J / rho / ratio / flags (and the seeded tables and moments) are bit-equal between the
paths, and the card's name and power limit. Not part of the product."""
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

MODES = {"pair": None, "one": "0"}
SEED_SAMPLES = 1


def set_mode(mode):
    if MODES[mode] is None:
        os.environ.pop("LQMPC_K1_PAIR", None)
    else:
        os.environ["LQMPC_K1_PAIR"] = MODES[mode]


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
    calls = {"batch": lambda: eng.eval_batch(dA, dB, x0, N, N),
             "seeded": lambda: eng.eval_seeded(SEED_SAMPLES, 0, S, 0.01, 0.01, N, N,
                                               want=("J", "rho", "ratio", "flags", "moments"))}
    res = {}
    for mode in MODES:
        set_mode(mode)
        for entry, call in calls.items():
            r = call()
            torch.cuda.synchronize()
            keys = ("J", "rho", "ratio", "flags") + (("moments",) if entry == "seeded" else ())
            res[mode, entry] = {k: r[k].cpu().numpy().copy() for k in keys}
    same = {"%s.%s" % (entry, k): bool(np.array_equal(res["pair", entry][k].view(np.uint8),
                                                       res["one", entry][k].view(np.uint8)))
            for entry in calls for k in res["pair", entry]}
    times = {(mode, entry): [] for mode in MODES for entry in calls}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for entry, call in calls.items():
            for mode in MODES:
                set_mode(mode)
                for _ in range(3):
                    call()
                e0.record()
                for _ in range(args.launches):
                    call()
                e1.record()
                torch.cuda.synchronize()
                times[mode, entry].append(e0.elapsed_time(e1) / args.launches)
    set_mode("pair")
    stat = lambda v: {"mean": float(np.mean(v)), "min": float(np.min(v)), "max": float(np.max(v)), "rounds": v}  # noqa: E731
    out = {"workload": "cfg-synth-4-2-10 K1 alone", "samples": S, "card": card(),
           "ms_per_launch": {entry: {mode: stat(times[mode, entry]) for mode in MODES} for entry in calls},
           "speedup": {entry: float(np.mean(times["one", entry]) / np.mean(times["pair", entry])) for entry in calls},
           "bit_equal": all(same.values()), "bit_equal_per_output": same}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
