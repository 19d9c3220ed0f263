"""Worst-case model error of the unconstrained law: sample, then ascend.

`worst_case_search` evaluates K1's performance ratio J_inf / V_expert(x0) on every sampled perturbation, takes the
`top_k` largest as starts and runs the projected ascent of `Engine.worst_case_batch` from each over the error set
{||dA|| <= e_A, ||dB|| <= e_B}. Sampling alone rarely lands near the worst case of a many-dimensional error set; the
ascent moves each start to a stationary point of J_inf on the set (or to an error that destabilises the loop).

`worst_case_search_sup` does the same without an x0: its objective is the worst ratio over every initial state,
gamma = lambda_max(S, P_exp), and its ascent is the joint one over the model error and the initial state.

`worst_case_search_inf` searches the input-constrained closed loop instead: its objective is K2c's certified J_inf of
the MPC law that re-solves the box-constrained QP every step (Engine.simulate_inf_batch), from a given initial state.

The operands are the engine's SoA layout: the grids `sampling.device_error_grids` returns (one error level, norm
'f' or '2') or `sampling.synth_samples_soa` draws (norm 'max'). Every step runs on the device.
"""
from __future__ import annotations

from .engine import FLAG_TAIL_UNCERTIFIED, FLAG_UNSTABLE


def worst_case_search(engine, dA, dB, x0, N: int, e_A: float, e_B: float, norm: str, top_k: int = 256,
                      max_iter: int = 200, tol: float = 1e-8):
    """dA [n*n][S], dB [n*m][S]; x0 [n][S] or one shared state [n]. Returns a dict:
      sampled_max_ratio, sampled_argmax: K1's largest ratio over the S samples and its index;
      per start (ordered by sampled ratio, +inf first, ties to the lowest index), device tensors: start_index,
        ratio_start, ratio, J, dA [n*n][k], dB [n*m][k], iters, flags;
      best_ratio, best_index: the largest ascended ratio and the sample index it started from;
      n_unstable: ascents that found a destabilising error in the set (ratio = +inf)."""
    torch = engine.torch
    n = engine.n
    dA, dB = engine._dev(dA), engine._dev(dB)
    S = dA.shape[-1]
    x0 = engine._dev(x0)
    if x0.numel() == n and S != 1:
        x0 = x0.reshape(n, 1).expand(n, S).contiguous()
    ratio = engine.eval_batch(dA, dB, x0, N, N, want=("ratio",))["ratio"][0]
    key = torch.nan_to_num(ratio, nan=-float("inf"), posinf=float("inf"))
    order = torch.sort(key, descending=True, stable=True).indices
    k = min(int(top_k), S)
    idx = order[:k]
    res = engine.worst_case_batch(dA[:, idx], dB[:, idx], x0[:, idx], N, e_A, e_B, norm, max_iter, tol)
    best = int(torch.argmax(torch.nan_to_num(res["ratio"], nan=-float("inf"))).item()) if k else -1
    return {
        "sampled_max_ratio": float(key[order[0]].item()) if S else float("nan"),
        "sampled_argmax": int(order[0].item()) if S else -1,
        "start_index": idx, "ratio_start": ratio[idx], "ratio": res["ratio"], "J": res["J"], "dA": res["dA"],
        "dB": res["dB"], "iters": res["iters"], "flags": res["flags"],
        "best_ratio": float(res["ratio"][best].item()) if k else float("nan"),
        "best_index": int(idx[best].item()) if k else -1,
        "n_unstable": int(((res["flags"] & FLAG_UNSTABLE) != 0).sum().item()),
    }


def worst_case_search_sup(engine, dA, dB, N: int, e_A: float, e_B: float, norm: str, top_k: int = 256,
                          max_iter: int = 200, tol: float = 1e-8):
    """worst_case_search over every initial state at once: ranks the S samples by gamma = sup_x0 J_inf / V_expert
    (Engine.ratio_sup_batch, value only; +inf first, ties to the lowest index) and runs the ascent of gamma
    (Engine.worst_case_sup_batch) from the `top_k` largest. dA [n*n][S], dB [n*m][S]. Returns the keys of
    worst_case_search with `ratio` (and sampled_max_ratio, ratio_start, best_ratio) meaning gamma and `J` = gamma (the
    cost J_inf(x_worst), since x_worst'P_exp x_worst = 1), plus x_worst [n][k]: the initial state attaining gamma."""
    torch = engine.torch
    dA, dB = engine._dev(dA), engine._dev(dB)
    S = dA.shape[-1]
    gamma = engine.ratio_sup_batch(dA, dB, N)["gamma"]
    key = torch.nan_to_num(gamma, nan=-float("inf"), posinf=float("inf"))
    order = torch.sort(key, descending=True, stable=True).indices
    k = min(int(top_k), S)
    idx = order[:k]
    res = engine.worst_case_sup_batch(dA[:, idx], dB[:, idx], N, e_A, e_B, norm, max_iter, tol)
    best = int(torch.argmax(torch.nan_to_num(res["gamma"], nan=-float("inf"))).item()) if k else -1
    return {
        "sampled_max_ratio": float(key[order[0]].item()) if S else float("nan"),
        "sampled_argmax": int(order[0].item()) if S else -1,
        "start_index": idx, "ratio_start": gamma[idx], "ratio": res["gamma"], "J": res["gamma"], "dA": res["dA"],
        "dB": res["dB"], "iters": res["iters"], "flags": res["flags"], "x_worst": res["x_worst"],
        "best_ratio": float(res["gamma"][best].item()) if k else float("nan"),
        "best_index": int(idx[best].item()) if k else -1,
        "n_unstable": int(((res["flags"] & FLAG_UNSTABLE) != 0).sum().item()),
    }


def worst_case_search_inf(engine, dA, dB, N: int, e_A: float, e_B: float, norm: str, x0=None, x0_shared=None,
                          top_k: int = 256, T_max: int = 1000, max_iter: int = 200, tol: float = 1e-8):
    """worst_case_search for the input-constrained closed loop: ranks the S samples by K2c's J_inf
    (Engine.simulate_inf_batch; +inf first, NaN last, ties to the lowest index) and runs the ascent of J_inf
    (Engine.worst_case_inf_batch) from the `top_k` largest. dA [n*n][S], dB [n*m][S]; x0 [n][S] or x0_shared (n,).
    Returns a dict with the keys of worst_case_search, J in place of the ratio:
      sampled_max_J, sampled_argmax: the largest sampled J_inf and its index;
      per start, device tensors: start_index, J_start, J, T_cert, dA [n*n][k], dB [n*m][k], iters, flags;
      best_J, best_index: the largest ascended J_inf and the sample index it started from;
      n_unstable: ascents that found a destabilising error (J = +inf);
      n_uncertified: samples whose J_inf was not certified within T_max steps (NaN, ranked last)."""
    torch = engine.torch
    dA, dB = engine._dev(dA), engine._dev(dB)
    S = dA.shape[-1]
    x0_sel = None if x0 is None else engine._dev(x0)
    v = engine.simulate_inf_batch(dA, dB, N, T_max, x0_shared=x0_shared, x0=x0_sel)
    J = v["J_inf"]
    key = torch.nan_to_num(J, nan=-float("inf"), posinf=float("inf"), neginf=-float("inf"))
    nan_last = torch.isnan(J).to(torch.int8)                 # NaN after every number, -inf included
    order = torch.sort(key, descending=True, stable=True).indices
    order = order[torch.sort(nan_last[order], stable=True).indices]
    k = min(int(top_k), S)
    idx = order[:k]
    res = engine.worst_case_inf_batch(dA[:, idx], dB[:, idx], N, e_A, e_B, norm, max_iter, tol, T_max,
                                      x0_shared=x0_shared, x0=None if x0_sel is None else x0_sel[:, idx])
    best = int(torch.argmax(torch.nan_to_num(res["J_inf"], nan=-float("inf"))).item()) if k else -1
    return {
        "sampled_max_J": float(J[order[0]].item()) if S else float("nan"),
        "sampled_argmax": int(order[0].item()) if S else -1,
        "start_index": idx, "J_start": J[idx], "J": res["J_inf"], "T_cert": res["T_cert"], "dA": res["dA"],
        "dB": res["dB"], "iters": res["iters"], "flags": res["flags"],
        "best_J": float(res["J_inf"][best].item()) if k else float("nan"),
        "best_index": int(idx[best].item()) if k else -1,
        "n_unstable": int(((res["flags"] & FLAG_UNSTABLE) != 0).sum().item()),
        "n_uncertified": int(((v["flags"] & FLAG_TAIL_UNCERTIFIED) != 0).sum().item()),
    }
