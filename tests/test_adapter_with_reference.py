"""The plugin boundary: `tinygp_b200.adapter.DirectSolver / QuasisepSolver` take tinygp's own kernel and noise objects
and must give what the reference computes with its own solvers.  tests/golden/adapter_vectors.npz holds, for every
case, the reference's results and its kernel / noise objects recorded as data (class name, module, field values;
made by tests/golden/make_golden_adapter.py, which also checks the reference's gp.py driving these solvers).  Here the
recorded objects are rebuilt as plain attribute holders of the same class and module names, so the adapter translates
exactly what it is given by tinygp, and a GaussianProcess drives the adapter's solvers.  The host layer runs over the
mock C-ABI (tests/hostmock.py), so no GPU is needed."""

import json
import os
import sys
from ctypes import c_void_p

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "golden"))

import adaptercases as C  # noqa: E402
import hostmock  # noqa: E402
from tinygp_b200 import GaussianProcess, _cabi, adapter, noise  # noqa: E402

GOLD = np.load(os.path.join(HERE, "golden", "adapter_vectors.npz"))
TREES = json.loads(str(GOLD["trees"]))
DENSE, QS = C.DENSE, C.QS


def foreign(node):
    """a recorded reference object: same class name, module and field values, no behaviour of its own"""
    if isinstance(node, list):
        return [foreign(v) for v in node]
    if not isinstance(node, dict):
        return node
    if "array" in node:
        return GOLD[node["array"]]
    obj = type(node["class"], (), {"__module__": node["module"]})()
    for name, value in node["fields"].items():
        setattr(obj, name, foreign(value))
    return obj


def objects(case):
    return {name: foreign(tree) for name, tree in TREES[case].items()}


@pytest.fixture()
def mock_device():
    lib = hostmock.MockLib()
    ctx = _cabi.Context.__new__(_cabi.Context)
    ctx.lib, ctx.handle, ctx.device = lib, c_void_p(1), -1
    previous = _cabi._ctx
    _cabi.set_context(ctx)
    try:
        yield
    finally:
        _cabi.set_context(previous)


def _close(a, key, tol=1e-9):
    a, b = np.asarray(a, dtype=np.float64), GOLD[key]
    assert a.shape == b.shape and np.all(np.isfinite(b)), "the reference itself must be finite for this comparison"
    assert np.max(np.abs(a - b)) <= tol * max(1.0, np.max(np.abs(b))), (key, np.max(np.abs(a - b)))


@pytest.mark.parametrize("expr", DENSE)
def test_reference_gaussian_process_with_b200_direct_solver(mock_device, expr):
    p = f"dense{DENSE.index(expr)}/"
    X, Xt, y = C.dense_inputs()
    ref = objects(p[:-1])
    ours = GaussianProcess(adapter.translate_kernel(ref["kernel"]), X, diag=0.07, mean=0.2, solver=adapter.DirectSolver)
    assert isinstance(ours.solver, adapter.DirectSolver)
    _close(ours.log_probability(y), p + "log_probability")
    _close(ours.variance, p + "variance")
    _close(ours.covariance, p + "covariance")
    lp_o, cond_o = ours.condition(y, Xt, diag=1e-3)
    _close(lp_o, p + "cond_log_probability")
    _close(cond_o.loc, p + "cond_loc")
    _close(cond_o.variance, p + "cond_variance")        # the Conditioned kernel calls back into our solve_triangular
    _close(cond_o.covariance, p + "cond_covariance")
    _close(cond_o.log_probability(np.cos(Xt[:, 0])), p + "cond_log_probability_test")
    mu_o, var_o = ours.predict(y, return_var=True)
    _close(mu_o, p + "predict_mean")
    _close(var_o, p + "predict_var")
    _close(ours.sample(C.SAMPLE_SEED, shape=C.SAMPLE_SHAPE), p + "sample")
    # the solver as tinygp's gp.py constructs and calls it: reference kernel and noise objects in, arrays out
    solver = adapter.DirectSolver(ref["kernel"], X, ref["noise"])
    _close(solver.covariance(), p + "covariance")
    _close(solver.variance(), p + "variance")
    _close(solver.normalization(), p + "normalization")
    _close(solver.condition(ref["kernel"], Xt, ref["test_noise"]), p + "solver_condition")


@pytest.mark.parametrize("expr", QS)
def test_reference_gaussian_process_with_b200_quasisep_solver(mock_device, expr):
    p = f"qs{QS.index(expr)}/"
    t, tt, y = C.qs_inputs()
    ref = objects(p[:-1])
    k = adapter.translate_kernel(ref["kernel"])
    ours = GaussianProcess(k, t, diag=0.07, solver=adapter.QuasisepSolver, parallel=True)
    _close(ours.log_probability(y), p + "log_probability")
    _close(ours.variance, p + "variance")
    lp_o, cond_o = ours.condition(y, tt, diag=1e-3)
    _close(lp_o, p + "cond_log_probability")
    _close(cond_o.loc, p + "cond_loc")
    _close(cond_o.variance, p + "cond_variance")
    # tinygp's gp.py takes the conditioned variance as kernel(X) + noise.diagonal() (solvers/direct.py:49), the
    # Conditioned kernel calling back into our solve_triangular
    _close(cond_o.kernel(tt) + cond_o.noise.diagonal(), p + "cond_variance")
    _close(cond_o.covariance, p + "cond_covariance")
    solver = adapter.QuasisepSolver(ref["kernel"], t, ref["noise"], parallel=True)
    _close(solver.variance(), p + "variance")
    _close(solver.normalization(), p + "normalization")
    _close(solver.condition(ref["kernel"], tt, ref["test_noise"]), p + "solver_condition")
    with pytest.raises(ValueError, match="Input coordinates must be sorted"):
        GaussianProcess(k, t[::-1].copy(), diag=0.07, solver=adapter.QuasisepSolver)


def test_unsupported_objects_are_refused_loudly(mock_device):
    X = np.linspace(0, 1, 5)
    with pytest.raises(NotImplementedError, match="unsupported by the B200"):
        adapter.DirectSolver(objects("unsupported")["kernel"], X, noise.Diagonal(np.full(5, 0.1)))


def test_reference_gaussian_process_with_banded_and_dense_noise(mock_device):
    """the reference's own noise.Banded / noise.Dense objects (noise.py:98-240) through the adapter's solvers"""
    t, tt, y, _, _ = C.banded_inputs()
    for j, solver in enumerate((adapter.QuasisepSolver, adapter.DirectSolver, adapter.DirectSolver)):
        p, ref = f"noise{j}/", objects(f"noise{j}")
        ours = GaussianProcess(adapter.translate_kernel(ref["kernel"]), t, noise=adapter.translate_noise(ref["noise"]),
                               solver=solver)
        _close(ours.log_probability(y), p + "log_probability")
        _close(ours.covariance, p + "covariance")
        lp_o, cond_o = ours.condition(y, tt, diag=1e-3)
        _close(lp_o, p + "cond_log_probability")
        _close(cond_o.loc, p + "cond_loc")
        _close(cond_o.covariance, p + "cond_covariance")
        s = solver(ref["kernel"], t, ref["noise"])
        _close(s.covariance(), p + "covariance")
        _close(s.normalization(), p + "normalization")
