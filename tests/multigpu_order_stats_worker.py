"""Worker of tests/test_order_stats_gpu.py::test_nccl_sharded_order_statistics_equal_single_gpu (one process per GPU
under torch.distributed.run, NCCL): quantiles and arg-extremes of a sharded 10^6 + 3-sample K1 table are bit-identical
on every rank and equal to the single-GPU result (rank 0 evaluates the whole set alone)."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

QS = (0.0, 0.05, 1 / 3, 0.5, 0.95, 0.999999, 1.0)


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from lq_mpc_b200 import sampling as sp, stats
    from lq_mpc_b200.engine import Engine
    eng = Engine(local)
    S = 1_000_003
    A, B, Q, R = sp.synth_problem(4, 2, seed=0)
    eng.set_problem(A, B, Q, R, Q, None, None, 30)
    lo, hi = stats.shard_bounds(S, rank, world)
    dA, dB, x0 = sp.synth_samples_soa(4, 2, hi - lo, seed=3, first=lo, e=0.05)
    r = eng.eval_batch(dA, dB, x0, 9, 10, want=("J", "rho", "ratio"))
    qv = stats.column_quantiles(eng, r["table"], QS)
    ax = stats.column_argext(eng, r["table"])                     # index_base: the prefix sum of shard lengths
    mine = torch.tensor(np.concatenate([qv.ravel().view(np.int64)] + [np.asarray(ax[k]).view(np.int64)
                                                                      for k in ("max", "argmax", "min", "argmin")]),
                        device="cuda")
    allm = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(allm, mine)
    for other in allm:
        assert torch.equal(other, allm[0]), "ranks disagree on the order statistics"
    if rank == 0:
        fA, fB, fx = sp.synth_samples_soa(4, 2, S, seed=3, first=0, e=0.05)
        full = eng.eval_batch(fA, fB, fx, 9, 10, want=("J", "rho", "ratio"))
        counts = eng.column_moments_raw(full["table"])[:, 2]          # the same protocol without collectives
        keys = stats.radix_select_keys(counts, stats.check_quantiles(QS),
                                       lambda pre, p: eng.column_radix_histogram_raw(full["table"], pre, p),
                                       lambda h: None, eng.column_radix_select_raw)
        single_q = stats.finish_quantiles(keys.cpu().numpy(), counts.cpu().numpy(), QS)
        single_a = stats.merge_argext(stats.pack_argext(*eng.column_argext_raw(full["table"])).cpu().numpy()[None])
        assert np.array_equal(qv.view(np.int64), single_q.view(np.int64))
        for k in single_a:
            assert np.array_equal(ax[k], single_a[k]), k
        tab = full["table"].cpu().numpy()
        for c in range(tab.shape[0]):
            f = tab[c][stats.k5_finite(tab[c])]
            assert np.array_equal(qv[:, c], np.quantile(f, QS)), c
        print("MULTIGPU_ORDER_STATS_OK world=%d S=%d unstable=%d" % (world, S, int((~np.isfinite(tab[0])).sum())),
              flush=True)
    dist.barrier()
    dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
