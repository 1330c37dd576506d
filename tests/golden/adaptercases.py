"""Cases of tests/test_adapter_with_reference.py, shared with make_golden_adapter.py (which runs them through the
reference's own GaussianProcess and records adapter_vectors.npz).  Inputs are regenerated from fixed seeds."""

import numpy as np

DENSE = [
    "1.7 * kernels.ExpSquared(0.9)",
    "kernels.Matern32(1.3, distance=kernels.L2Distance()) + 0.3 * kernels.RationalQuadratic(scale=1.5, alpha=0.8)",
    "kernels.Exp(1.3) * kernels.ExpSquared(3.0) + 0.05",
    "transforms.Subspace(0, kernels.ExpSquared(1.2)) + 0.5 * transforms.Linear(np.array([0.7, 1.4]), kernels.Matern52(0.9))",
]

QS = [
    "quasisep.SHO(omega=1.5, quality=3.0, sigma=1.8) + quasisep.Matern32(scale=1.5, sigma=0.9)",
    "2.0 * quasisep.Matern52(1.2) + quasisep.Celerite(1.1, 0.1, 0.3, 1.5)",
    "quasisep.Cosine(scale=3.0, sigma=0.7) + quasisep.Exp(scale=2.0, sigma=0.5)",
]

SAMPLE_SEED, SAMPLE_SHAPE = 4, (3,)


def dense_inputs():
    rng = np.random.default_rng(3)
    X, Xt = rng.uniform(0, 4, (40, 2)), rng.uniform(0, 4, (6, 2))
    y = np.sin(X[:, 0]) + 0.1 * rng.normal(size=40)
    return X, Xt, y


def qs_inputs():
    rng = np.random.default_rng(5)
    t = np.sort(rng.uniform(0, 12, 60))
    tt = rng.uniform(-1, 13, 5)
    y = np.sin(t) + 0.1 * rng.normal(size=60)
    return t, tt, y


def banded_inputs():
    """coordinates, test coordinates, data, and the diagonal / off-diagonals of a banded noise model"""
    rng = np.random.default_rng(8)
    t = np.sort(rng.uniform(0, 12, 50))
    tt, y = rng.uniform(-1, 13, 5), np.sin(t)
    diag, off_diags = rng.uniform(0.1, 0.2, 50), 0.02 * rng.normal(size=(50, 2))
    return t, tt, y, diag, off_diags


def sample_normals(num_data):
    """the standard normal draws behind GaussianProcess.sample(SAMPLE_SEED, shape=SAMPLE_SHAPE)"""
    return np.random.default_rng(SAMPLE_SEED).standard_normal((num_data,) + SAMPLE_SHAPE)
