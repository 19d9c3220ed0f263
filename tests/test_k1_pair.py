"""K1 with two samples per thread (one horizon, n <= 4) against the one-sample kernel (LQMPC_K1_PAIR=0).

The two-sample kernel runs each sample's operation sequence unchanged, only interleaved with a second sample's, so every
output must be bit-identical, not merely close: J, rho, ratio, flags, V_N, J_T and K0 of eval_batch, and the tables and
moments of eval_seeded. Batch sizes straddle the 128-sample halves of a 256-sample CTA, so the second slot of a thread is
present, absent (it then computes on the first slot's operands and stores nothing) and absent in a partial last CTA.
Among the samples are unstable closed loops, one placed so that it lands in a tail slot, and, in a separate case, samples
whose Cholesky factor fails at the first Riccati step.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PAIR_DIMS = [(1, 1), (2, 1), (2, 2), (3, 1), (3, 2), (3, 3), (4, 1), (4, 2), (4, 4)]
SIZES = [1, 127, 128, 129, 255, 256, 257, 100_003]
N_HOR, T_SIM = 6, 7


def _bit_equal(a, b):
    import torch
    if a.dtype == torch.float64:
        a, b = a.view(torch.int64), b.view(torch.int64)
    return a.shape == b.shape and torch.equal(a, b)


def _samples(rng, A, B, S):
    """SoA operands: small model errors, plus sign-flipped input gains (unstable closed loops) at a few indices, the
    last sample among them; for S = 200 that one sits in the second slot of a thread, and sample 127, whose partner
    s0 + 128 = 255 lies past the end, sits in a thread with an empty second slot."""
    n, m = B.shape
    dA = rng.uniform(-0.05, 0.05, size=(S, n, n))
    dB = rng.uniform(-0.05, 0.05, size=(S, n, m))
    x0 = rng.normal(size=(S, n))
    for s in {0, S // 3, 127 % S, S - 1}:
        dB[s] = -2.5 * B
    return dA, dB, x0


def _run(engine, dA, dB, x0, pair, monkeypatch):
    import torch
    from oracle import np_batched as nb
    if pair:
        monkeypatch.delenv("LQMPC_K1_PAIR", raising=False)
    else:
        monkeypatch.setenv("LQMPC_K1_PAIR", "0")
    soa = [torch.from_numpy(a).cuda() for a in nb.to_soa(dA, dB, x0)]
    got = engine.eval_batch(*soa, N_HOR, N_HOR, T=T_SIM, want=("J", "rho", "ratio", "V_N", "J_T", "flags", "K0"))
    torch.cuda.synchronize()
    return got


@pytest.mark.parametrize("n,m", PAIR_DIMS)
def test_pair_kernel_bit_equal_to_one_sample_kernel(engine, n, m, monkeypatch):
    from oracle import np_batched as nb
    A, B, Q, R = nb.synth_problem(n, m, seed=10 * n + m)
    engine.set_problem(A, B, Q, R, Q, None, None, 30)
    rng = np.random.default_rng(n * 100 + m)
    unstable_seen = 0
    for S in SIZES + [200]:
        dA, dB, x0 = _samples(rng, A, B, S)
        one = _run(engine, dA, dB, x0, False, monkeypatch)
        two = _run(engine, dA, dB, x0, True, monkeypatch)
        for k in ("J", "rho", "ratio", "V_N", "J_T", "flags", "K0"):
            assert _bit_equal(one[k], two[k]), (S, k)
        unstable_seen += int(np.count_nonzero(one["flags"].cpu().numpy() & 1))
    assert unstable_seen > 0          # the sign-flipped gains do destabilise closed loops


@pytest.mark.parametrize("n,m", [(2, 1), (3, 2), (4, 2), (4, 4)])
def test_pair_kernel_sticky_cholesky_flag(engine, n, m, monkeypatch):
    """An indefinite terminal weight makes R + B^' P B^ indefinite at the first step for samples with a large B^."""
    from oracle import np_batched as nb
    A, B, Q, R = nb.synth_problem(n, m, seed=3)
    engine.set_problem(A, B, Q, R, -0.02 * np.eye(n), None, None, 30)
    rng = np.random.default_rng(5)
    S = 300
    dA, dB, x0 = _samples(rng, A, B, S)
    bad = [5, 140, 299]
    for s in bad:
        dB[s] = 20.0 * np.ones((n, m))
    one = _run(engine, dA, dB, x0, False, monkeypatch)
    two = _run(engine, dA, dB, x0, True, monkeypatch)
    for k in ("J", "rho", "ratio", "V_N", "J_T", "flags", "K0"):
        assert _bit_equal(one[k], two[k]), k
    fl = two["flags"].cpu().numpy()[0]
    assert all(fl[s] & 256 for s in bad)


@pytest.mark.parametrize("n,m", PAIR_DIMS)
def test_pair_seeded_kernel_bit_equal(engine, n, m, monkeypatch):
    from oracle import np_batched as nb
    A, B, Q, R = nb.synth_problem(n, m, seed=n + 7 * m)
    engine.set_problem(A, B, Q, R, Q, None, None, 30)
    for S, first in ((1, 0), (129, 5), (257, (1 << 32) - 100), (100_003, 12_345)):
        res = []
        for pair in (False, True):
            if pair:
                monkeypatch.delenv("LQMPC_K1_PAIR", raising=False)
            else:
                monkeypatch.setenv("LQMPC_K1_PAIR", "0")
            res.append(engine.eval_seeded(9, first, S, 0.05, 0.05, N_HOR, N_HOR,
                                          want=("J", "rho", "ratio", "flags", "moments")))
        for k in ("table", "flags", "moments"):
            assert _bit_equal(res[0][k], res[1][k]), (S, k)
