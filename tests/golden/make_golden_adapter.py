"""Generate tests/golden/adapter_vectors.npz: the UNMODIFIED reference `tinygp.GaussianProcess` (dfm/tinygp sources
found by refimport.py, over the NumPy stand-ins of tests/golden/jaxshim) on the cases of adaptercases.py, with its own
solvers.  Besides the results, every reference kernel and noise object is recorded as data (class name, module and
field values), so that the test can hand the adapter objects shaped like tinygp's without the reference present.
Before writing, the same reference GaussianProcess is run with solver=tinygp_b200.adapter.* over the mock C-ABI
(tests/hostmock.py) and must reproduce every recorded value.  Run from the repo root:
python tests/golden/make_golden_adapter.py
"""

import dataclasses
import json
import os
import sys
from ctypes import c_void_p

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import adaptercases as C  # noqa: E402
import refimport  # noqa: E402


def record(obj, arrays, key):
    """a reference object as JSON-able data; arrays go to `arrays` under `key`"""
    if getattr(type(obj), "__is_shim_module__", False):
        return {"class": type(obj).__name__, "module": type(obj).__module__,
                "fields": {f.name: record(getattr(obj, f.name), arrays, f"{key}.{f.name}")
                           for f in dataclasses.fields(obj)}}
    if isinstance(obj, (np.ndarray, np.generic)):
        if np.ndim(obj) == 0:
            return obj.item()
        arrays[key] = np.asarray(obj)
        return {"array": key}
    if obj is None or isinstance(obj, (bool, int, float, str)):
        return obj
    if isinstance(obj, (tuple, list)):
        return [record(v, arrays, f"{key}.{i}") for i, v in enumerate(obj)]
    raise TypeError(f"cannot record {type(obj).__name__} at {key}")


def sample_value(gp):
    """a sample by the formula of gp.py's sample(), mean + L z, mirrored here with the normals of
    adaptercases.sample_normals (the reference draws its own from jax.random); only L z = dot_triangular(z) is the
    reference's"""
    z = C.sample_normals(gp.num_data)
    return np.asarray(gp.mean) + np.moveaxis(np.asarray(gp.solver.dot_triangular(z)), 0, -1)


def main():
    tinygp = refimport.install()
    from tinygp import GaussianProcess, kernels, noise, transforms
    from tinygp.kernels import quasisep
    from tinygp.solvers import DirectSolver, QuasisepSolver

    arrays, trees = {}, {}

    def put(prefix, **values):
        for name, v in values.items():
            arrays[f"{prefix}/{name}"] = np.asarray(v, dtype=np.float64)

    def objects(prefix, **objs):
        trees[prefix] = {name: record(o, arrays, f"{prefix}/{name}") for name, o in objs.items()}

    X, Xt, y = C.dense_inputs()
    for i, expr in enumerate(C.DENSE):
        k = eval(expr, {"kernels": kernels, "transforms": transforms, "np": np})
        gp = GaussianProcess(k, X, diag=0.07, mean=0.2)
        lp_c, cond = gp.condition(y, Xt, diag=1e-3)
        mu, var = gp.predict(y, return_var=True)
        test_noise = noise.Diagonal(diag=np.full(len(Xt), 1e-3))
        p = f"dense{i}"
        objects(p, kernel=k, noise=gp.noise, test_noise=test_noise)
        put(p, log_probability=gp.log_probability(y), variance=gp.variance, covariance=gp.covariance,
            cond_log_probability=lp_c, cond_loc=cond.loc, cond_variance=cond.variance, cond_covariance=cond.covariance,
            cond_log_probability_test=cond.log_probability(np.cos(Xt[:, 0])), predict_mean=mu, predict_var=var,
            sample=sample_value(gp), normalization=gp.solver.normalization(),
            solver_condition=gp.solver.condition(k, Xt, test_noise))

    t, tt, y = C.qs_inputs()
    for i, expr in enumerate(C.QS):
        k = eval(expr, {"quasisep": quasisep})
        gp = GaussianProcess(k, t, diag=0.07)
        lp_c, cond = gp.condition(y, tt, diag=1e-3)
        test_noise = noise.Diagonal(diag=np.full(len(tt), 1e-3))
        p = f"qs{i}"
        objects(p, kernel=k, noise=gp.noise, test_noise=test_noise)
        put(p, log_probability=gp.log_probability(y), variance=gp.variance, cond_log_probability=lp_c,
            cond_loc=cond.loc, cond_variance=cond.variance, cond_covariance=cond.covariance,
            normalization=gp.solver.normalization(), solver_condition=gp.solver.condition(k, tt, test_noise))

    t, tt, y, diag, off_diags = C.banded_inputs()
    banded = noise.Banded(diag=diag, off_diags=off_diags)
    dense = noise.Dense(value=np.asarray(banded + np.zeros((50, 50))))
    kq = quasisep.Matern32(scale=1.5, sigma=1.8) + quasisep.Exp(scale=0.7)
    combos = ((kq, banded, QuasisepSolver), (kq, banded, DirectSolver), (kernels.Matern52(1.1), dense, DirectSolver))
    for j, (k, nz, solver) in enumerate(combos):
        gp = GaussianProcess(k, t, noise=nz, solver=solver)
        lp_c, cond = gp.condition(y, tt, diag=1e-3)
        p = f"noise{j}"
        objects(p, kernel=k, noise=nz)
        put(p, log_probability=gp.log_probability(y), covariance=gp.covariance, cond_log_probability=lp_c,
            cond_loc=cond.loc, cond_covariance=cond.covariance, normalization=gp.solver.normalization())
    objects("unsupported", kernel=kernels.DotProduct())

    check_adapter_under_reference(tinygp, arrays)
    meta = {"generator": "tests/golden/make_golden_adapter.py",
            "reference": "dfm/tinygp sources executed over tests/golden/jaxshim (NumPy %s)" % np.__version__}
    out = os.path.join(HERE, "adapter_vectors.npz")
    np.savez_compressed(out, trees=np.array(json.dumps(trees)), meta=np.array(json.dumps(meta)), **arrays)
    print("wrote", out, os.path.getsize(out), "bytes")


def check_adapter_under_reference(tinygp, arrays, tol=1e-9):
    """the reference's gp.py driving tinygp_b200.adapter's solvers (host layer over the mock C-ABI) must reproduce
    what it computes with its own solvers"""
    import hostmock
    from tinygp_b200 import _cabi, adapter
    from tinygp import GaussianProcess, kernels, noise, transforms
    from tinygp.kernels import quasisep

    ctx = _cabi.Context.__new__(_cabi.Context)
    ctx.lib, ctx.handle, ctx.device = hostmock.MockLib(), c_void_p(1), -1
    _cabi.set_context(ctx)

    def close(a, key):
        b = arrays[key]
        a = np.asarray(a, dtype=np.float64)
        assert a.shape == b.shape and np.max(np.abs(a - b)) <= tol * max(1.0, np.max(np.abs(b))), key

    X, Xt, y = C.dense_inputs()
    for i, expr in enumerate(C.DENSE):
        k = eval(expr, {"kernels": kernels, "transforms": transforms, "np": np})
        gp = GaussianProcess(k, X, diag=0.07, mean=0.2, solver=adapter.DirectSolver)
        lp_c, cond = gp.condition(y, Xt, diag=1e-3)
        for name, v in (("log_probability", gp.log_probability(y)), ("covariance", gp.covariance),
                        ("cond_log_probability", lp_c), ("cond_covariance", cond.covariance),
                        ("cond_variance", cond.variance), ("sample", sample_value(gp))):
            close(v, f"dense{i}/{name}")
    t, tt, y = C.qs_inputs()
    for i, expr in enumerate(C.QS):
        gp = GaussianProcess(eval(expr, {"quasisep": quasisep}), t, diag=0.07, solver=adapter.QuasisepSolver,
                             parallel=True)
        lp_c, cond = gp.condition(y, tt, diag=1e-3)
        for name, v in (("log_probability", gp.log_probability(y)), ("variance", gp.variance),
                        ("cond_log_probability", lp_c), ("cond_covariance", cond.covariance)):
            close(v, f"qs{i}/{name}")
    t, tt, y, diag, off_diags = C.banded_inputs()
    banded = noise.Banded(diag=diag, off_diags=off_diags)
    gp = GaussianProcess(quasisep.Matern32(scale=1.5, sigma=1.8) + quasisep.Exp(scale=0.7), t, noise=banded,
                         solver=adapter.QuasisepSolver)
    close(gp.log_probability(y), "noise0/log_probability")
    print("reference GaussianProcess with the adapter's solvers reproduces the reference's own solvers")


if __name__ == "__main__":
    main()
