"""CPU tier — how often the closed-form spectral radius of eig.cuh (n = 3, 4: characteristic polynomial -> Ferrari
start -> Bairstow refinement -> acceptance test) is trusted, and how accurate it is where it is. Everything it rejects
goes to the QR iteration, so a lower acceptance rate costs time, not accuracy; these pins keep a change to the starting
point or the refinement from quietly moving work onto the QR path. Same families and seeds as
test_hostmath.py::test_closed_form_spectral_radius_is_trusted_only_when_accurate."""
import numpy as np
import pytest

from oracle import np_batched as nb

hm = pytest.importorskip("tests.hostmath.api")

# acceptance rates of the double-precision Ferrari start with three Bairstow steps on these seeds
ACCEPTED = {3: {"gauss": 1.0000, "scaled": 0.9957, "sym": 1.0000, "cluster": 0.9446, "huge_range": 1.0000},
            4: {"gauss": 1.0000, "scaled": 0.9960, "sym": 1.0000, "cluster": 0.0216, "huge_range": 1.0000}}


def _families(n):
    rng = np.random.default_rng(10 + n)
    S = 60_000
    return {"gauss": rng.normal(size=(S, n, n)),
            "scaled": rng.normal(size=(S, n, n)) * np.exp(rng.uniform(-3, 3, size=(S, n, 1))),
            "sym": (lambda M: M + M.transpose(0, 2, 1))(rng.normal(size=(S, n, n))),
            "cluster": 0.9 * np.eye(n)[None] + 0.02 * rng.normal(size=(S, n, n)),
            "tight": 0.9 * np.eye(n)[None] + 1e-3 * rng.normal(size=(S, n, n)),
            "huge_range": rng.normal(size=(S, n, n)) * 10.0 ** rng.integers(-100, 100, size=(S, 1, 1))}


@pytest.mark.parametrize("n", [3, 4])
def test_closed_form_acceptance_rates_hold(n):
    for name, M in _families(n).items():
        rho, ok = hm.spectral_radius_poly(M)
        tr = ok == 1
        if name == "tight":
            assert tr.mean() < 0.01, (name, tr.mean())
        else:
            assert tr.mean() >= ACCEPTED[n][name] - 0.001, (name, tr.mean())
        ref = np.max(np.abs(np.linalg.eigvals(M[tr])), axis=1)
        if tr.any():
            assert np.max(np.abs(rho[tr] - ref) / ref) < 1e-10, name


@pytest.mark.parametrize("e", [0.01, 0.3])
def test_closed_form_takes_every_headline_closed_loop(e):
    """The flagship distribution (synthetic (4, 2) plant, N = 10, model errors U[-e, e]): every closed loop A + B K_0
    of the estimated-model gain is accepted by the closed form and agrees with LAPACK to 1e-12."""
    n, m, N, S = 4, 2, 10, 100_000
    A, B, Q, R = nb.synth_problem(n, m, seed=0)
    dA, dB, x0 = nb.synth_samples(n, m, S, seed=1, e=e)
    got = hm.eval_batch(A, B, Q, R, Q, 30, *nb.to_soa(dA, dB, x0), N, N, 0)
    K = got["K0"][0].reshape(m, n, S).transpose(2, 0, 1)
    Acl = A[None] + B[None] @ K
    rho, ok = hm.spectral_radius_poly(Acl)
    assert np.all(ok == 1), int(np.sum(ok != 1))
    ref = np.max(np.abs(np.linalg.eigvals(Acl)), axis=1)
    assert np.max(np.abs(rho - ref) / ref) < 1e-12
    assert np.max(np.abs(got["rho"][0] - ref) / ref) < 1e-12      # and so does the engine's K1 math
