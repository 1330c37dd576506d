"""The __host__ __device__ core of the quasiseparable CUDA path (tinygp_b200/csrc/qs_core.cuh: model lowering,
per-point generators `qs_gen`, the `GramBack` scan monoid and its chunk / tree / replay decomposition) compiled for
the CPU by tests/csrc/qs_hostcheck.cu and compared with the oracle.  Same source as the kernels; what is NOT covered
here is the launch geometry and memory system, which the `-m gpu` tests cover."""

import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import tinygp_np as o
from tinygp_b200.kernels import quasisep as Q

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "csrc", "qs_hostcheck.cu")
OUT = os.path.join(HERE, "csrc", "_build", "libqs_hostcheck.so")
DEPS = [SRC, os.path.join(HERE, "..", "tinygp_b200", "csrc", "qs_core.cuh"),
        os.path.join(HERE, "..", "tinygp_b200", "csrc", "qs_fast.cuh"),
        os.path.join(HERE, "..", "tinygp_b200", "csrc", "common.cuh")]

KERNELS = {
    "sho+m32": (Q.SHO(1.5, 3.0, 1.8) + Q.Matern32(1.5, 0.9), o.qs.SHO(1.5, 3.0, 1.8) + o.qs.Matern32(1.5, 0.9)),
    "sho_critical": (Q.SHO(1.2, 0.5, 1.1), o.qs.SHO(1.2, 0.5, 1.1)),
    "sho_overdamped": (Q.SHO(1.2, 0.2, 1.1), o.qs.SHO(1.2, 0.2, 1.1)),
    "exp": (Q.Exp(1.7, 0.8), o.qs.Exp(1.7, 0.8)),
    "m52": (Q.Matern52(2.5, 1.3), o.qs.Matern52(2.5, 1.3)),
    "celerite": (Q.Celerite(1.1, 0.1, 0.3, 1.5), o.qs.Celerite(1.1, 0.1, 0.3, 1.5)),
    "cosine+exp": (Q.Cosine(3.0, 0.7) + Q.Exp(2.0, 0.5), o.qs.Cosine(3.0, 0.7) + o.qs.Exp(2.0, 0.5)),
    "product_sho_m32": (Q.SHO(1.5, 3.0, 1.8) * Q.Matern32(1.5, 0.9), o.qs.SHO(1.5, 3.0, 1.8) * o.qs.Matern32(1.5, 0.9)),
    "scaled_product_plus_m52": (0.7 * (Q.Exp(2.0, 1.1) * Q.Celerite(1.1, 0.1, 0.3, 1.5)) + Q.Matern52(2.5, 1.3),
                                o.qs.Scale(o.qs.Exp(2.0, 1.1) * o.qs.Celerite(1.1, 0.1, 0.3, 1.5), 0.7) + o.qs.Matern52(2.5, 1.3)),
    "carma31+m32": (Q.CARMA(np.array([1.4, 2.3, 1.5]), np.array([0.1, 0.5])) + 0.5 * Q.Matern32(1.5),
                    o.qs.CARMA(np.array([1.4, 2.3, 1.5]), np.array([0.1, 0.5])) + o.qs.Scale(o.qs.Matern32(1.5, 1.0), 0.5)),
    "carma21_complex": (Q.CARMA(np.array([1.0, 1.2]), np.array([1.0, 3.0])), o.qs.CARMA(np.array([1.0, 1.2]), np.array([1.0, 3.0]))),
    "carma21_real": (Q.CARMA(np.array([0.1, 1.1]), np.array([1.0, 3.0])), o.qs.CARMA(np.array([0.1, 1.1]), np.array([1.0, 3.0]))),
    # a Sum inside a Product is multiplied out by the host layer: two Kronecker-structured terms, block after block
    "product_of_sum_multiplied_out": ((Q.Matern32(1.5, 0.9) + 0.4 * Q.Exp(0.7)) * Q.SHO(1.5, 3.0, 1.8),
                                      o.qs.Matern32(1.5, 0.9) * o.qs.SHO(1.5, 3.0, 1.8)
                                      + o.qs.Scale(o.qs.Exp(0.7, 1.0), 0.4) * o.qs.SHO(1.5, 3.0, 1.8)),
    "product_carma_pair_first": (Q.CARMA(np.array([1.0, 1.2]), np.array([1.0, 3.0])) * Q.Exp(2.0, 1.1),
                                 o.qs.CARMA(np.array([1.0, 1.2]), np.array([1.0, 3.0])) * o.qs.Exp(2.0, 1.1)),
    # 7 and 8 states, the largest the backend compiles (B200GP_QS_MAX_J)
    "product_m52_cosine+exp_7": (Q.Matern52(2.5, 1.3) * Q.Cosine(3.0, 0.7) + Q.Exp(2.0, 0.5),
                                 o.qs.Matern52(2.5, 1.3) * o.qs.Cosine(3.0, 0.7) + o.qs.Exp(2.0, 0.5)),
    "m52+m52+sho_8": (Q.Matern52(2.5, 1.3) + Q.Matern52(0.6, 0.4) + Q.SHO(1.5, 3.0, 0.8),
                      o.qs.Matern52(2.5, 1.3) + o.qs.Matern52(0.6, 0.4) + o.qs.SHO(1.5, 3.0, 0.8)),
    "scaled_sum3": (2.0 * Q.Matern32(1.2) + Q.SHO(0.8, 4.0, 0.6) + 0.5 * Q.Exp(5.0),
                    o.qs.Scale(o.qs.Matern32(1.2, 1.0), 2.0) + o.qs.SHO(0.8, 4.0, 0.6) + o.qs.Scale(o.qs.Exp(5.0, 1.0), 0.5)),
}


@pytest.fixture(scope="module")
def lib():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    if not os.path.exists(OUT) or any(os.path.getmtime(d) > os.path.getmtime(OUT) for d in DEPS):
        os.makedirs(os.path.dirname(OUT), exist_ok=True)
        tmp = f"{OUT}.{os.getpid()}"     # parallel workers each build their own copy and swap it in whole
        subprocess.run([nvcc, "-O2", "-std=c++17", "-Wno-deprecated-gpu-targets", "-Xcompiler", "-fPIC", "-shared",
                        "-o", tmp, SRC], check=True)
        os.replace(tmp, OUT)
    return ctypes.CDLL(OUT)


def _p(a):
    return ctypes.c_void_p(a.ctypes.data)


def _data(n, seed=0, ties=True):
    rng = np.random.default_rng(seed)
    t = np.sort(rng.uniform(0, n / 8.0, n))
    if ties and n > 10:
        t[7] = t[6]
    return t, rng.uniform(0.05, 0.2, n)


@pytest.mark.parametrize("name", list(KERNELS))
def test_model_and_generators_match_the_oracle(lib, name):
    """build_model + qs_gen (kernels/quasisep.py:102-116 and the state-space models :343-673)"""
    k, ko = KERNELS[name]
    comps = k.component_array()
    t, _ = _data(200)
    d, p, q, a = ko.to_symm_qsm(t)
    J = ctypes.c_int()
    qm, hm, d0 = np.zeros(8), np.zeros(8), ctypes.c_double()
    assert lib.hostcheck_model(_p(comps), comps.shape[0], ctypes.byref(J), _p(qm), _p(hm), ctypes.byref(d0)) == 0
    assert J.value == p.shape[1] == k.state_dim()
    np.testing.assert_allclose(qm[:J.value], q[0], rtol=1e-14, atol=1e-15)
    np.testing.assert_allclose(d0.value, d[0], rtol=1e-14)
    ad, pd = np.zeros(a.shape), np.zeros(p.shape)      # (zeros_like would copy the oracle's swapped strides)
    assert lib.hostcheck_generators(_p(comps), comps.shape[0], _p(t), ctypes.c_int64(t.size), _p(ad), _p(pd)) == 0
    np.testing.assert_allclose(ad, a, rtol=1e-13, atol=1e-15)
    np.testing.assert_allclose(pd, p, rtol=1e-13, atol=1e-15)


@pytest.mark.parametrize("chunk", [1, 7, 64])
@pytest.mark.parametrize("n", [1, 5, 300, 5000])
@pytest.mark.parametrize("name", ["sho+m32", "m52", "exp", "scaled_sum3"])
def test_inverse_diagonal_scan_matches_the_oracle(lib, name, n, chunk):
    """diag((K + N)^-1) by the GramBack scan: chunk composites, the fan-in-16 tree (two levels at n = 5000, chunk 1)
    and the replay give the diagonal of the dense inverse"""
    k, ko = KERNELS[name]
    comps = k.component_array()
    t, noise = _data(n, seed=n)
    s = o.QuasisepSolver(ko, t, o.Diagonal(noise))
    out = np.zeros(n)
    c, w = np.ascontiguousarray(s.c), np.ascontiguousarray(s.w)
    assert lib.hostcheck_inverse_diagonal(_p(comps), comps.shape[0], _p(t), ctypes.c_int64(n), _p(c), _p(w), chunk,
                                          _p(out)) == 0
    if n <= 300:
        want = np.diag(np.linalg.inv(s.covariance()))
    else:   # columns of L^-1 by the oracle's sequential solve: (Sigma^-1)_ii = |L^-1 e_i|^2 on a sample of columns
        idx = np.unique(np.r_[0, 1, n // 2, n - 2, n - 1, np.random.default_rng(1).integers(0, n, 12)])
        E = np.zeros((n, idx.size)); E[idx, np.arange(idx.size)] = 1.0
        Z = s.solve_triangular(s.solve_triangular(E), transpose=True)      # Sigma^-1 e_i
        want, out = Z[idx, np.arange(idx.size)], out[idx]
    np.testing.assert_allclose(out, want, rtol=1e-10, atol=0)


# ------------------------------------------------------------------------------------------------
# dense path: the kernel-program interpreter (kprog.cuh) on the CPU against the REFERENCE's kernel values
# ------------------------------------------------------------------------------------------------
KSRC = os.path.join(HERE, "csrc", "kprog_hostcheck.cu")
KOUT = os.path.join(HERE, "csrc", "_build", "libkprog_hostcheck.so")
KDEPS = [KSRC, os.path.join(HERE, "..", "tinygp_b200", "csrc", "kprog.cuh"),
         os.path.join(HERE, "..", "tinygp_b200", "csrc", "common.cuh"), os.path.join(HERE, "..", "include", "b200gp.h")]


@pytest.fixture(scope="module")
def klib():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    if not os.path.exists(KOUT) or any(os.path.getmtime(d) > os.path.getmtime(KOUT) for d in KDEPS):
        os.makedirs(os.path.dirname(KOUT), exist_ok=True)
        tmp = f"{KOUT}.{os.getpid()}"
        subprocess.run([nvcc, "-O2", "-std=c++17", "-Wno-deprecated-gpu-targets", "-diag-suppress", "20013",
                        "-Xcompiler", "-fPIC", "-shared", "-o", tmp, KSRC], check=True)
        os.replace(tmp, KOUT)
    return ctypes.CDLL(KOUT)


def _kmat(klib, k, X1, X2):
    prog, x1 = k.lower_for(X1)
    _, x2 = k.lower_for(X2)
    out, err = np.empty((x1.shape[0], x2.shape[0])), ctypes.create_string_buffer(256)
    rc = klib.hostcheck_kernel_matrix(_p(prog), prog.shape[0], _p(x1), ctypes.c_int64(x1.shape[0]), _p(x2),
                                      ctypes.c_int64(x2.shape[0]), x1.shape[1], _p(out), err)
    assert rc == 0, err.value
    return out


def _kmat_fast(klib, k, X1, X2):
    prog, x1 = k.lower_for(X1)
    _, x2 = k.lower_for(X2)
    out, err = np.empty((x1.shape[0], x2.shape[0])), ctypes.create_string_buffer(256)
    rc = klib.hostcheck_kernel_matrix_fast(_p(prog), prog.shape[0], _p(x1), ctypes.c_int64(x1.shape[0]), _p(x2),
                                           ctypes.c_int64(x2.shape[0]), x1.shape[1], _p(out), err)
    assert rc in (0, 4), err.value
    return out if rc == 0 else None


def _dense_cases():
    import sys
    sys.path.insert(0, os.path.join(HERE, "golden"))
    import refcases
    return [c for c in refcases.CASES if c["kind"] == "dense"], refcases


@pytest.mark.parametrize("case", _dense_cases()[0], ids=[c["name"] for c in _dense_cases()[0]])
def test_kernel_program_interpreter_reproduces_reference_kernel_values(klib, case):
    """Kernel.__call__ (base.py:84-103) for every stationary leaf / distance default / sum / product / transform of the
    golden set: host lowering (Kernel.lower_for) + the device interpreter source, against the reference's numbers"""
    import json
    from test_reference_golden import product_namespace
    refcases = _dense_cases()[1]
    gold = json.load(open(os.path.join(HERE, "golden", "reference_vectors.json")))["cases"][case["name"]]
    if "K_cross" not in gold:
        pytest.skip("non-PD case: the reference returned -inf before any kernel values were recorded")
    inp = refcases._inputs(case)
    k = product_namespace().kernel(case["kernel"])
    idx = np.arange(0, case["n"], max(1, case["n"] // 9))[:9]
    got = _kmat(klib, k, inp["X"][idx], inp["X_test"])
    np.testing.assert_allclose(got, np.array(gold["K_cross"]), rtol=1e-13, atol=1e-15)
    fast = _kmat_fast(klib, k, inp["X"][idx], inp["X_test"])      # sum-of-products normal form (None: program has none)
    if fast is not None:
        np.testing.assert_allclose(fast, np.array(gold["K_cross"]), rtol=1e-13, atol=1e-15)
    else:
        assert "transforms" in case["kernel"] or "Subspace" in case["kernel"] or "Linear" in case["kernel"] \
            or "Cholesky" in case["kernel"], case["kernel"]
    prog, x = k.lower_for(inp["X"][idx])
    d, err = ctypes.c_double(), ctypes.create_string_buffer(256)
    assert klib.hostcheck_kernel_diag(_p(prog), prog.shape[0], x.shape[1], ctypes.byref(d), err) == 0, err.value
    np.testing.assert_allclose(np.full(idx.size, d.value), np.array(gold["K_diag"]), rtol=1e-14)


@pytest.mark.parametrize("name", ["sho+m32", "sho_critical", "sho_overdamped", "exp", "m52", "celerite", "cosine+exp",
                                  "scaled_sum3"])
def test_quasisep_closed_forms_through_the_interpreter(klib, name):
    """dense evaluation of a quasiseparable kernel (kernels/quasisep.py:118-145) = its tau program in the same
    interpreter, against the oracle's state-space evaluate"""
    k, ko = KERNELS[name]
    rng = np.random.default_rng(4)
    t1, t2 = rng.uniform(0, 12, 9), rng.uniform(0, 12, 7)
    t2[0] = t1[0]
    np.testing.assert_allclose(_kmat(klib, k, t1, t2), ko(t1, t2), rtol=1e-12, atol=1e-14)


def test_malformed_programs_are_rejected_by_the_parser(klib):
    X = np.zeros((2, 2))
    out, err = np.empty((2, 2)), ctypes.create_string_buffer(256)

    def run(rows):
        prog = np.ascontiguousarray(np.array(rows, dtype=np.float64))
        return klib.hostcheck_kernel_matrix(_p(prog), prog.shape[0], _p(X), ctypes.c_int64(2), _p(X), ctypes.c_int64(2), 2,
                                            _p(out), err), err.value.decode()

    assert run([[2, 1, 1.0, 0]])[0] == 0
    assert "stack underflow" in run([[16, 0, 0, 0]])[1]
    assert "malformed" in run([[2, 1, 1.0, 0], [2, 1, 1.0, 0]])[1]
    assert "unknown opcode" in run([[11, 0, 1.0, 0]])[1]
    assert "undefined metric" in run([[2, 3, 1.0, 0]])[1]
    assert "width does not match" in run([[32, 1, 1, 3], [1, 0, 0, 0], [2, 3, 1.0, 0]])[1]
    assert "non-finite" in run([[32, 1, 1, 2], [np.nan, 0, 0, 0], [2, 3, 1.0, 0]])[1]


# ------------------------------------------------------------------------------------------------
# the Cholesky and affine scans of the quasiseparable path (BASELINE config 4's hot kernels) on the CPU
# ------------------------------------------------------------------------------------------------
OPS = {"lower_solve": 0, "upper_solve": 1, "lower_dot": 2, "symm_lower": 3, "symm_upper": 4}


def _factor(lib, k, t, noise, chunk, x=None):
    comps = k.component_array()
    n, J = t.size, k.state_dim()
    c, w = np.zeros(n), np.zeros((n, J))
    ld, info = ctypes.c_double(), ctypes.c_int()
    alpha = np.zeros(n) if x is not None else None
    rc = lib.hostcheck_factor(_p(comps), comps.shape[0], _p(t), _p(noise), ctypes.c_int64(n), chunk, _p(c), _p(w),
                              ctypes.byref(ld), ctypes.byref(info), _p(x) if x is not None else None,
                              _p(alpha) if x is not None else None)
    assert rc == 0
    return c, w, ld.value, info.value, alpha


@pytest.mark.parametrize("chunk", [1, 5, 64])
@pytest.mark.parametrize("n", [1, 3, 257, 4100])
@pytest.mark.parametrize("name", list(KERNELS))
def test_cholesky_scan_matches_the_sequential_recursion(lib, name, n, chunk):
    """chol_chunk_body -> Riccati tree -> chol_replay_body (ops.py:352-399): c, w, sum log c and the fused forward
    solve equal the oracle's sequential recursion (ops.py:354-361, 465-468)"""
    k, ko = KERNELS[name]
    t, noise = _data(n, seed=n + 1)
    y = np.sin(t)
    so = o.QuasisepSolver(ko, t, o.Diagonal(noise))
    c, w, ld, info, alpha = _factor(lib, k, t, noise, chunk, x=y)
    assert info == 0
    np.testing.assert_allclose(c, so.c, rtol=1e-11, atol=0)
    np.testing.assert_allclose(w, so.w, rtol=1e-10, atol=1e-13)
    np.testing.assert_allclose(ld, np.sum(np.log(so.c)), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(alpha, so.solve_triangular(y), rtol=1e-9, atol=1e-12)


def test_cholesky_scan_reports_the_first_bad_pivot(lib):
    k, ko = KERNELS["sho+m32"]
    t, noise = _data(300)
    bad = noise.copy()
    bad[123] = -50.0
    c, w, ld, info, _ = _factor(lib, k, t, bad, 16)
    d, p, q, a = ko.to_symm_qsm(t)
    _, _, first = __import__("oracle.cref", fromlist=["x"]).qs_cholesky(d + bad, p, q, a)
    assert info == first and info >= 1


@pytest.mark.parametrize("chunk", [1, 7, 64])
@pytest.mark.parametrize("n", [1, 258, 3000])
@pytest.mark.parametrize("name", ["sho+m32", "m52", "cosine+exp"])
def test_affine_scans_match_the_oracle(lib, name, n, chunk):
    """triangular solves and products (ops.py:308-349, 463-512; core.py:303-305, 499-505) as chunk / tree / replay"""
    k, ko = KERNELS[name]
    comps = k.component_array()
    t, noise = _data(n, seed=n + 2)
    rng = np.random.default_rng(n)
    x = rng.normal(size=n)
    so = o.QuasisepSolver(ko, t, o.Diagonal(noise))
    c, w = np.ascontiguousarray(so.c), np.ascontiguousarray(so.w)

    def run(op, out=None):
        out = np.zeros(n) if out is None else out
        assert lib.hostcheck_affine(_p(comps), comps.shape[0], OPS[op], _p(t), _p(noise), _p(c), _p(w), _p(x),
                                    ctypes.c_int64(n), chunk, _p(out)) == 0
        return out

    np.testing.assert_allclose(run("lower_solve"), so.solve_triangular(x), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(run("upper_solve"), so.solve_triangular(x, transpose=True), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(run("lower_dot"), so.dot_triangular(x), rtol=1e-10, atol=1e-12)
    ky = run("symm_upper", run("symm_lower"))            # K y = (d y + lower part) + upper part
    if n <= 300:
        np.testing.assert_allclose(ky, so.covariance() @ x, rtol=1e-10, atol=1e-11)
    else:
        lo = o.qs_lower_matmul(so.p, so.q, so.a, x[:, None])[:, 0]
        up = o.qs_upper_matmul(so.p, so.q, so.a, x[:, None])[:, 0]
        np.testing.assert_allclose(ky, so.d * x + lo + up, rtol=1e-10, atol=1e-11)


@pytest.mark.parametrize("case", _dense_cases()[0], ids=[c["name"] for c in _dense_cases()[0]])
def test_parsed_programs_re_encode_to_the_same_rows(klib, case):
    """kprog_encode (used when a parsed program crosses the C-ABI again: the streaming factorisation of very large N)
    must reproduce the host lowering row for row -- including the metric definitions of input transforms"""
    from test_reference_golden import product_namespace
    refcases = _dense_cases()[1]
    k = product_namespace().kernel(case["kernel"])
    prog, x = k.lower_for(refcases._inputs(case)["X"][:4])
    out = np.zeros((prog.shape[0] + 4, 4))
    n = klib.hostcheck_reencode(_p(prog), prog.shape[0], x.shape[1], _p(out), out.shape[0])
    assert n == prog.shape[0]
    np.testing.assert_array_equal(out[:n], prog)


@pytest.mark.parametrize("n,chunk", [(40, 1), (1100, 1), (33000, 1), (5000, 7)])
def test_warp_scan_tree_gives_the_same_states(lib, n, chunk):
    """option qs_tree = 1 (warp-shuffle Hillis-Steele scan over the chunk composites, fan-in 32; 1, 2 and 3 levels here):
    the emulation of that algorithm with the device monoids reproduces the oracle for the Cholesky (Riccati), the solves
    (Affine) and the inverse diagonal (GramBack)"""
    k, ko = KERNELS["sho+m32"]
    comps = k.component_array()
    t, noise = _data(n, seed=n + 7)
    x = np.sin(t)
    so = o.QuasisepSolver(ko, t, o.Diagonal(noise))
    lib.hostcheck_set_tree(1)
    try:
        c, w, ld, info, alpha = _factor(lib, k, t, noise, chunk, x=x)
        out = np.zeros(n)
        assert lib.hostcheck_affine(_p(comps), comps.shape[0], OPS["upper_solve"], _p(t), _p(noise), _p(c), _p(w), _p(x),
                                    ctypes.c_int64(n), chunk, _p(out)) == 0
        inv = np.zeros(n)
        assert lib.hostcheck_inverse_diagonal(_p(comps), comps.shape[0], _p(t), ctypes.c_int64(n), _p(c), _p(w), chunk,
                                              _p(inv)) == 0
    finally:
        lib.hostcheck_set_tree(0)
    assert info == 0
    np.testing.assert_allclose(c, so.c, rtol=1e-10, atol=0)
    np.testing.assert_allclose(w, so.w, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(alpha, so.solve_triangular(x), rtol=1e-8, atol=1e-11)
    np.testing.assert_allclose(out, so.solve_triangular(x, transpose=True), rtol=1e-8, atol=1e-11)
    idx = np.unique(np.r_[0, n // 2, n - 1])
    E = np.zeros((n, idx.size)); E[idx, np.arange(idx.size)] = 1.0
    want = so.solve_triangular(so.solve_triangular(E), transpose=True)[idx, np.arange(idx.size)]
    np.testing.assert_allclose(inv[idx], want, rtol=1e-9, atol=0)


# ------------------------------------------------------------------------------------------------
# the layout-specialised fast path (qs_fast.cuh): same checks, plus sum of squares without a third pass
# ------------------------------------------------------------------------------------------------
FAST_KERNELS = dict(KERNELS)
FAST_KERNELS.update({
    "celerite+m52": (Q.Celerite(1.1, 0.1, 0.3, 1.5) + Q.Matern52(2.5, 1.3),
                     o.qs.Celerite(1.1, 0.1, 0.3, 1.5) + o.qs.Matern52(2.5, 1.3)),
    "exp+exp+m32": (Q.Exp(1.7, 0.8) + Q.Exp(0.6, 0.4) + Q.Matern32(2.0, 0.7),
                    o.qs.Exp(1.7, 0.8) + o.qs.Exp(0.6, 0.4) + o.qs.Matern32(2.0, 0.7)),
    "sho3": (Q.SHO(1.5, 3.0, 1.8) + Q.SHO(0.4, 0.2, 0.5) + Q.SHO(2.2, 0.5, 0.3),
             o.qs.SHO(1.5, 3.0, 1.8) + o.qs.SHO(0.4, 0.2, 0.5) + o.qs.SHO(2.2, 0.5, 0.3)),
})


@pytest.mark.parametrize("name", list(FAST_KERNELS))
def test_fast_generators_match_the_oracle(lib, name):
    """qsf_gen (compile-time block offsets, host-prepared reciprocals) against kernels/quasisep.py:102-116"""
    k, ko = FAST_KERNELS[name]
    comps = k.component_array()
    t, _ = _data(200)
    d, p, q, a = ko.to_symm_qsm(t)
    ad, pd = np.zeros(a.shape), np.zeros(p.shape)
    rc = lib.hostcheck_fast_generators(_p(comps), comps.shape[0], _p(t), ctypes.c_int64(t.size), _p(ad), _p(pd))
    if "product" in name or name.endswith("_8"):
        assert rc == 4          # Kronecker-structured terms / 8 states have no specialised layout: generic kernels
        return
    assert rc == 0
    np.testing.assert_allclose(ad, a, rtol=1e-13, atol=1e-15)
    np.testing.assert_allclose(pd, p, rtol=1e-13, atol=1e-15)


@pytest.mark.parametrize("tree", [0, 1])
@pytest.mark.parametrize("chunk", [1, 5, 64])
@pytest.mark.parametrize("n", [1, 3, 257, 4100])
@pytest.mark.parametrize("name", list(FAST_KERNELS))
def test_fast_factor_and_fused_sum_of_squares(lib, name, n, chunk, tree):
    """qsf_chunk_body -> tree -> qsf_replay_body -> tree -> qsf_quad_eval: c, w, sum log c of ops.py:354-361 and
    |L^-1 y|^2 (gp.py:313-316) from the per-chunk quadratic sums, no forward-substitution pass over the points"""
    k, ko = FAST_KERNELS[name]
    comps = k.component_array()
    t, noise = _data(n, seed=n + 1)
    y = np.sin(t) + 0.3 * np.cos(3.1 * t)
    so = o.QuasisepSolver(ko, t, o.Diagonal(noise))
    J = k.state_dim()
    c, w = np.zeros(n), np.zeros((n, J))
    ld, info, ss = ctypes.c_double(), ctypes.c_int(), ctypes.c_double()
    lib.hostcheck_set_tree(tree)
    try:
        rc = lib.hostcheck_fast_factor(_p(comps), comps.shape[0], _p(t), _p(noise), ctypes.c_int64(n), chunk, _p(c), _p(w),
                                       ctypes.byref(ld), ctypes.byref(info), _p(y), ctypes.byref(ss))
    finally:
        lib.hostcheck_set_tree(0)
    if "product" in name or name.endswith("_8"):
        assert rc == 4
        return
    assert rc == 0 and info.value == 0
    np.testing.assert_allclose(c, so.c, rtol=1e-11, atol=0)
    np.testing.assert_allclose(w, so.w, rtol=1e-10, atol=1e-13)
    np.testing.assert_allclose(ld.value, np.sum(np.log(so.c)), rtol=1e-12, atol=1e-12)
    alpha = so.solve_triangular(y)
    np.testing.assert_allclose(ss.value, np.sum(alpha ** 2), rtol=1e-10)


def test_fast_factor_reports_the_first_bad_pivot(lib):
    k = Q.SHO(1.5, 3.0, 1.8) + Q.Matern32(1.5, 0.9)
    comps = k.component_array()
    n = 500
    t, noise = _data(n, seed=3)
    noise = noise.copy()
    noise[321] = -50.0                                     # makes the pivot at 321 negative
    c, w = np.zeros(n), np.zeros((n, 4))
    ld, info, ss = ctypes.c_double(), ctypes.c_int(), ctypes.c_double()
    y = np.sin(t)
    assert lib.hostcheck_fast_factor(_p(comps), comps.shape[0], _p(t), _p(noise), ctypes.c_int64(n), 64, _p(c), _p(w),
                                     ctypes.byref(ld), ctypes.byref(info), _p(y), ctypes.byref(ss)) == 0
    assert info.value == 322                               # 1-based index of the first non-positive pivot


def test_normal_form_covers_the_benchmark_kernels_and_refuses_what_it_cannot_represent(klib):
    """kprog_to_fast: BASELINE configs 2 / 3 / 5 have a normal form; five leaves or five terms do not"""
    from tinygp_b200 import kernels
    rng = np.random.default_rng(5)
    X1, X2 = rng.uniform(0, 4, (7, 3)), rng.uniform(0, 4, (5, 3))
    L2 = kernels.L2Distance()
    ok = [1.0 * kernels.ExpSquared(1.0), 1.5 * kernels.Matern52(2.0, L2) + 0.7 * kernels.RationalQuadratic(1.5, L2, alpha=1.5),
          (kernels.Matern32(1.3, L2) + 0.2) * kernels.ExpSquared(0.8) * 2.5, kernels.Exp(1.1, L2) + kernels.Cosine(2.0, L2) * 0.3 + 0.01]
    for k in ok:
        fast = _kmat_fast(klib, k, X1, X2)
        assert fast is not None
        np.testing.assert_allclose(fast, _kmat(klib, k, X1, X2), rtol=2e-15, atol=0)
    e = kernels.ExpSquared(0.8)
    np.testing.assert_allclose(_kmat_fast(klib, e * e, X1, X2), _kmat(klib, e * e, X1, X2), rtol=2e-15, atol=0)
    five = kernels.ExpSquared(0.5) + kernels.ExpSquared(0.6) + kernels.ExpSquared(0.7) + kernels.ExpSquared(0.8) + kernels.ExpSquared(0.9)
    assert _kmat_fast(klib, five, X1, X2) is None
