"""Development probe (GPU box): K4 (n=32, m=8, N=30) parity vs the batched oracle + timing of the spectral-radius modes:
by squaring (default) / by the QR kernel for every sample. Not part of the product."""
import json, os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from lq_mpc_b200.engine import Engine
from oracle import np_batched as nb

eng = Engine(0)
n, m, N = 32, 8, 30
A, B, Q, R = nb.synth_problem(n, m, seed=0)
eng.set_problem_tiled(A, B, Q, R, Q, 30)
Pexp = nb.expert_matrix(A, B, Q, R, Q, 30)
print("Pexp err", float(np.max(np.abs(eng.prepared_tiled()["Pexp"] - Pexp) / np.abs(Pexp).max())))
dA, dB, x0 = nb.synth_samples(n, m, 512, seed=1, e=1e-3)
ref = nb.eval_batch(A, B, Q, R, Q, Pexp, dA, dB, x0, N, N)
out = {}
S = int(sys.argv[1]) if len(sys.argv) > 1 else 125_000
g = torch.Generator(device="cuda").manual_seed(0)
bA = (torch.rand((S, n, n), device="cuda", dtype=torch.float64, generator=g) - 0.5) * 2e-3
bB = (torch.rand((S, n, m), device="cuda", dtype=torch.float64, generator=g) - 0.5) * 2e-3
bx = torch.randn((S, n), device="cuda", dtype=torch.float64, generator=g)
rho_by = {}
for rho in ("sq", "qr"):
    os.environ["LQMPC_K4_RHO"] = rho
    got = eng.eval_batch_tiled(dA, dB, x0, N, N)
    errs = {k: float(np.max(np.abs(got[k].cpu().numpy() - ref[k]) / np.abs(ref[k]))) for k in ("J", "rho", "ratio")}
    for _ in range(2):
        eng.eval_batch_tiled(bA, bB, bx, N, N)
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    K = 3
    for _ in range(K):
        r = eng.eval_batch_tiled(bA, bB, bx, N, N)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / K
    rho_by[rho] = r["rho"].cpu().numpy()
    res = {"parity": errs, "flags": np.unique(got["flags"].cpu().numpy()).tolist(), "S": S, "ms": ms,
           "evals_per_s": S / (ms * 1e-3), "unstable": int((r["flags"] & 1).sum()),
           "flags_big": np.unique(r["flags"].cpu().numpy()).tolist()}
    tag = rho
    print(tag, json.dumps(res))
    out[tag] = res
d = np.abs(rho_by["sq"] - rho_by["qr"]) / rho_by["qr"]
out["rho_sq_vs_qr_max_rel"] = float(d.max())
print("rho squaring vs QR on the big batch: max rel diff", float(d.max()))
json.dump(out, open("gpurun_out/k4_probe.json", "w"), indent=1)
