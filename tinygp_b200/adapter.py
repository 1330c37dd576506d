"""Plug the B200 solvers into the REFERENCE's own ``tinygp.GaussianProcess`` as ``solver=``.

    import tinygp
    from tinygp_b200 import adapter
    gp = tinygp.GaussianProcess(tinygp.kernels.ExpSquared(1.5), X, diag=0.1, solver=adapter.DirectSolver)
    gp.log_probability(y)            # tinygp's gp.py drives; K build + Cholesky + solves run on the B200

``tinygp.GaussianProcess`` calls its solver as a constructor, ``solver(kernel, X, noise, covariance=..., **kw)``
(src/tinygp/gp.py:106-112), and then only through the six methods of ``solvers.solver.Solver``
(src/tinygp/solvers/solver.py:15-82).  The classes here honour exactly that contract with *reference* objects on
the outside: the kernel / noise passed in are tinygp's own equinox modules; they are translated, by class name and
field, into the parameter holders of ``tinygp_b200.kernels`` (which lower to the device kernel program), and every
method forwards to the C-ABI-backed solver of ``tinygp_b200.solvers``.

Scope: eager use.  tinygp decorates ``GaussianProcess._compute_log_prob`` etc. with ``jax.jit`` and traces ``self``,
so inside real JAX these classes additionally have to be ``equinox.Module``s whose methods go through
``jax.pure_callback`` (INTEGRATION.md section 3) -- JAX is not installable in this image, so that last wrapper is
not built; the Solver interface itself is exercised end to end by tests/golden/make_golden_adapter.py, which runs the
unmodified reference ``GaussianProcess`` with these solvers, and by tests/test_adapter_with_reference.py against its
recorded results.
"""

from __future__ import annotations

__all__ = ["DirectSolver", "QuasisepSolver", "translate_kernel", "translate_noise"]

from typing import Any

import numpy as np

from tinygp_b200 import kernels as K
from tinygp_b200 import noise as N
from tinygp_b200 import solvers as S
from tinygp_b200 import transforms as T
from tinygp_b200.kernels import quasisep as Q


def _f(x) -> float:
    return float(np.asarray(x))


def _is_quasisep(k) -> bool:
    return type(k).__module__.endswith("quasisep")


def translate_kernel(k) -> K.Kernel:
    """tinygp kernel pytree -> tinygp_b200 kernel (src/tinygp/kernels/{base,stationary,quasisep}.py, transforms.py)."""
    if isinstance(k, K.Kernel):
        return k
    name = type(k).__name__
    if _is_quasisep(k):
        if name == "Sum":
            return Q.Sum(translate_kernel(k.kernel1), translate_kernel(k.kernel2))
        if name == "Scale":
            return Q.Scale(translate_kernel(k.kernel), _f(k.scale))
        if name == "Celerite":
            return Q.Celerite(_f(k.a), _f(k.b), _f(k.c), _f(k.d))
        if name == "SHO":
            return Q.SHO(_f(k.omega), _f(k.quality), _f(k.sigma))
        if name in ("Exp", "Matern32", "Matern52", "Cosine"):
            return getattr(Q, name)(_f(k.scale), _f(k.sigma))
        raise NotImplementedError(f"quasiseparable kernel {name} is unsupported by the B200 solver backend")
    if name == "Sum":
        return K.Sum(translate_kernel(k.kernel1), translate_kernel(k.kernel2))
    if name == "Product":
        return K.Product(translate_kernel(k.kernel1), translate_kernel(k.kernel2))
    if name == "Constant":
        return K.Constant(_f(k.value))
    if name in ("Exp", "ExpSquared", "Matern32", "Matern52", "Cosine", "ExpSineSquared", "RationalQuadratic"):
        dname = type(k.distance).__name__
        if dname not in ("L1Distance", "L2Distance"):
            raise NotImplementedError("custom Distance metrics are unsupported by the B200 solver backend")
        dist = getattr(K, dname)()
        if name == "ExpSineSquared":
            return K.ExpSineSquared(_f(k.scale), dist, gamma=_f(k.gamma))
        if name == "RationalQuadratic":
            return K.RationalQuadratic(_f(k.scale), dist, alpha=_f(k.alpha))
        return getattr(K, name)(_f(k.scale), dist)
    if name == "Linear":
        return T.Linear(np.asarray(k.scale, dtype=np.float64), translate_kernel(k.kernel))
    if name == "Cholesky":
        return T.Cholesky(np.asarray(k.factor, dtype=np.float64), translate_kernel(k.kernel))
    if name == "Subspace":
        return T.Subspace(k.axis if np.ndim(k.axis) == 0 else np.asarray(k.axis), translate_kernel(k.kernel))
    if name == "Transform":
        return T.Transform(k.transform, translate_kernel(k.kernel))
    if name == "Conditioned":   # kernels/base.py:129-153: (X, solver, kernel); `solver` is one of the adapters below
        inner = k.solver.inner if isinstance(k.solver, _Adapter) else k.solver
        return K.Conditioned(np.asarray(k.X), inner, translate_kernel(k.kernel))
    raise NotImplementedError(f"kernel {name} is unsupported by the B200 solver backend")


def translate_noise(noise) -> N.Noise:
    """src/tinygp/noise.py:55-240"""
    if isinstance(noise, N.Noise):
        return noise
    if type(noise).__name__ == "Diagonal":
        return N.Diagonal(np.asarray(noise.diag, dtype=np.float64))
    if type(noise).__name__ == "Banded":      # noise.py:126-240
        return N.Banded(np.asarray(noise.diag, dtype=np.float64), np.asarray(noise.off_diags, dtype=np.float64))
    if type(noise).__name__ == "Dense":       # noise.py:98-123
        return N.Dense(np.asarray(noise.value, dtype=np.float64))
    raise NotImplementedError(f"noise model {type(noise).__name__} is unsupported by the B200 solver backend")


class _Adapter:
    """the six Solver methods (solvers/solver.py:40-82), forwarded"""

    inner: Any

    def variance(self):
        return self.inner.variance()

    def covariance(self):
        return self.inner.covariance()

    def normalization(self):
        return self.inner.normalization()

    def solve_triangular(self, y, *, transpose: bool = False):
        return self.inner.solve_triangular(np.asarray(y, dtype=np.float64), transpose=transpose)

    def dot_triangular(self, y):
        return self.inner.dot_triangular(np.asarray(y, dtype=np.float64))

    def condition(self, kernel, X_test, noise):
        Xt = None if X_test is None else np.asarray(X_test, dtype=np.float64)
        # asanyarray keeps the ConditionedCovariance tag that tinygp_b200.GaussianProcess reads for the variance
        return np.asanyarray(self.inner.condition(translate_kernel(kernel), Xt, translate_noise(noise)))


class DirectSolver(_Adapter):
    """drop-in for tinygp.solvers.DirectSolver (src/tinygp/solvers/direct.py:17-95)"""

    def __init__(self, kernel, X, noise, *, covariance: Any | None = None):
        cov = None if covariance is None else np.asarray(covariance, dtype=np.float64)
        self.X = X
        self.inner = S.DirectSolver(translate_kernel(kernel), np.asarray(X, dtype=np.float64), translate_noise(noise),
                                    covariance=cov)

    @classmethod
    def init(cls, kernel, X, noise, *, covariance: Any | None = None):   # solvers/solver.py:29-38
        return cls(kernel, X, noise, covariance=covariance)


class QuasisepSolver(_Adapter):
    """drop-in for tinygp.solvers.QuasisepSolver (src/tinygp/solvers/quasisep/solver.py:19-139)"""

    def __init__(self, kernel, X, noise, *, covariance: Any | None = None, assume_sorted: bool = False,
                 parallel: bool = False):
        self.X = X
        self.inner = S.QuasisepSolver(translate_kernel(kernel), np.asarray(X, dtype=np.float64), translate_noise(noise),
                                      covariance=covariance, assume_sorted=assume_sorted, parallel=parallel)

    @classmethod
    def init(cls, kernel, X, noise, *, covariance: Any | None = None, **kw):
        return cls(kernel, X, noise, covariance=covariance, **kw)
