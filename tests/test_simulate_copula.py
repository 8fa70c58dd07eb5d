"""Host side of the Gaussian-copula form of simulate_transcriptomes (reference memento/simulate.py:69-88): argument
checks that must fail before anything is drawn, the CUDA-only refusal on a CPU device, and the covariance factor."""
import numpy as np
import pytest
import torch

from memento_b200 import simulate

MEANS = np.array([0.5, 3.0, 20.0])
VARS = MEANS + 0.3 * MEANS ** 2


@pytest.mark.parametrize("cov, what", [
    (np.eye(2), "square with side G"),
    (np.ones((3, 2)), "square with side G"),
    (np.array([[1.0, 0.5, 0.0], [0.4, 1.0, 0.0], [0.0, 0.0, 1.0]]), "symmetric"),
    (np.array([[1.0, 2.0, 0.0], [2.0, 1.0, 0.0], [0.0, 0.0, 1.0]]), "positive semidefinite"),
    (np.diag([1.0, np.nan, 1.0]), "finite"),
])
def test_invalid_norm_cov_raises_value_error(cov, what):
    with pytest.raises(ValueError):
        simulate.simulate_transcriptomes(10, MEANS, VARS, norm_cov=cov, device="cpu")


@pytest.mark.parametrize("means, variances", [
    (np.array([0.5, 0.0, 2.0]), np.array([1.0, 1.0, 3.0])),          # a zero mean: r = 0
    (np.array([0.5, -1.0, 2.0]), np.array([1.0, 1.0, 3.0])),         # a negative mean
    (np.array([0.5, 2.0, 2.0]), np.array([1.0, 2.0, 3.0])),          # variance == mean: r = inf
    (np.array([0.5, np.nan, 2.0]), np.array([1.0, 1.0, 3.0])),
    (np.array([0.5, 1.0]), np.array([1.0, 2.0, 3.0])),               # lengths differ
])
def test_invalid_nb_parameters_raise_value_error(means, variances):
    with pytest.raises(ValueError):
        simulate.simulate_transcriptomes(10, means, variances, norm_cov=np.eye(len(means)), device="cpu")


def test_cpu_device_is_refused():
    with pytest.raises(NotImplementedError, match="CUDA"):
        simulate.simulate_transcriptomes(10, MEANS, VARS, norm_cov=np.eye(3), device="cpu")
    with pytest.raises(NotImplementedError, match="CUDA"):
        simulate.simulate_transcriptomes(10, MEANS, VARS, norm_cov=np.eye(3))


def test_factor_reproduces_psd_and_rank_deficient_matrices():
    rng = np.random.default_rng(3)
    a = rng.standard_normal((40, 40))
    full = a @ a.T / 40
    b = rng.standard_normal((40, 7))
    low = b @ b.T / 7                                        # rank 7
    latent1 = np.array([[1.0, 1.0, 0.0], [1.0, 1.0, 0.0], [0.0, 0.0, 2.0]])      # two genes at correlation 1
    for m in (full, low, latent1):
        f = simulate.copula_factor(m, "cpu")
        assert f.dtype == torch.float64 and f.shape == m.shape
        np.testing.assert_allclose((f @ f.T).numpy(), m, rtol=0, atol=1e-12)
    # eigenvalues at rounding level are dropped as scipy's multivariate_normal drops them
    assert int((simulate.copula_factor(low, "cpu").abs().sum(dim=0) > 0).sum()) == 7
    # slightly negative within scipy's tolerance is accepted
    w, v = np.linalg.eigh(low)
    w[0] = -1e-12
    simulate.copula_factor((v * w) @ v.T, "cpu")
