"""Development probe (GPU box): per-phase cycle counts of k4a. Needs the library built with
LQMPC_NVCC_EXTRA=-DLQ_K4_PROFILE (the launcher then prints `k4prof` lines to stderr). Not part of the product."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from lq_mpc_b200.engine import Engine
from oracle import np_batched as nb

eng = Engine(0)
n, m, N = 32, 8, 30
A, B, Q, R = nb.synth_problem(n, m, seed=0)
eng.set_problem_tiled(A, B, Q, R, Q, 30)
S = 125_000
g = torch.Generator(device="cuda").manual_seed(0)
bA = (torch.rand((S, n, n), device="cuda", dtype=torch.float64, generator=g) - 0.5) * 2e-3
bB = (torch.rand((S, n, m), device="cuda", dtype=torch.float64, generator=g) - 0.5) * 2e-3
bx = torch.randn((S, n), device="cuda", dtype=torch.float64, generator=g)
for _ in range(2):
    eng.eval_batch_tiled(bA, bB, bx, N, N)
torch.cuda.synchronize()
