"""CPU suite for the product's host side: the C ABI library loads and exports every symbol that
include/rebvo_b200.h declares, fails loudly without a GPU (no fallback), and its host/device algebra (lm.cuh)
agrees with the reference's TooN results and with numpy."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def test_abi_exports_every_declared_symbol(built):
    from rebvo_b200 import capi
    hdr = open(os.path.join(ROOT, "include", "rebvo_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = sorted(set(re.findall(r"\b(rb_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 40
    L = capi.lib()
    missing = [s for s in declared if not hasattr(L, s)]
    assert not missing, missing
    assert sorted(capi.SYMBOLS) == declared


def test_keyline_layout_is_the_reference_layout(built):
    from rebvo_b200 import capi
    from oracle import refapi
    assert capi.KEYLINE.itemsize == 168
    assert capi.KEYLINE == refapi.KEYLINE
    if refapi.available():
        assert refapi.lib().ref_sizeof_keyline() == 168


def test_no_silent_cpu_fallback(built):
    """Without a CUDA device the product must refuse to run (RB_ERR_NO_DEVICE), never fall back."""
    import torch
    from rebvo_b200 import capi, synth
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(capi.RbError):
        capi.Ctx(synth.EUROC, 3.56359, 1.2599)
    with pytest.raises(capi.RbError):
        capi.Pipeline(capi.default_params(synth.EUROC), max_batch=2)


def test_so3_against_reference_toon(built):
    from rebvo_b200 import capi
    from oracle import refapi
    L = capi.lib()
    rng = np.random.default_rng(0)
    ws = [np.zeros(3), np.array([1e-5, -2e-5, 3e-5]), np.array([4e-4, 1e-4, -6e-4]), np.array([0.01, -0.02, 0.005]),
          np.array([0.3, -1.2, 0.7]), np.array([2.0, 1.5, -1.0])] + [rng.normal(0, 0.5, 3) for _ in range(20)]
    for w in ws:
        R = np.zeros((3, 3))
        L.rb_hostmath_so3_exp(_p(w), _p(R))
        assert np.allclose(R @ R.T, np.eye(3), atol=1e-12)
        back = np.zeros(3)
        L.rb_hostmath_so3_ln(_p(R), _p(back))
        assert np.allclose(back, w, atol=1e-9), (w, back)
        if refapi.available():
            Rr = refapi.so3_exp(w)
            assert np.array_equal(R, Rr), "SO3::exp differs from TooN for %s" % w
            assert np.allclose(refapi.so3_ln(Rr), back, atol=1e-13)


def test_ldlt_and_pinv_solvers(built):
    from rebvo_b200 import capi
    L = capi.lib()
    rng = np.random.default_rng(1)
    for _ in range(20):
        J = rng.normal(size=(40, 6)) * rng.uniform(0.1, 100, 6)
        A = J.T @ J
        A = A + np.eye(6) * 1e-3 * A.max()
        b = rng.normal(size=6)
        x = np.zeros(6)
        L.rb_hostmath_chol6_solve(_p(A), _p(b), _p(x))
        assert np.allclose(x, np.linalg.solve(A, b), rtol=1e-9)
        L.rb_hostmath_solve_sym6_like_svd(_p(A), _p(b), _p(x))
        assert np.allclose(x, np.linalg.solve(A, b), rtol=1e-9)
        L.rb_hostmath_sym_svd_backsub(_p(A), 6, _p(b), _p(x))
        assert np.allclose(x, np.linalg.pinv(A, rcond=1e-9) @ b, rtol=1e-8)
        inv = np.zeros((6, 6))
        L.rb_hostmath_chol6_inverse(_p(A), _p(inv))
        assert np.allclose(inv, np.linalg.inv(A), rtol=1e-8)
    # rank deficient: pseudo-inverse semantics of SVD<>::backsub (condition 1e9)
    J = rng.normal(size=(40, 6))
    J[:, 5] = J[:, 0]
    A = J.T @ J
    b = A @ rng.normal(size=6)
    x = np.zeros(6)
    L.rb_hostmath_sym_svd_backsub(_p(A), 6, _p(b), _p(x))
    assert np.allclose(x, np.linalg.pinv(A, rcond=1e-9) @ b, rtol=1e-6, atol=1e-9)
    M = rng.normal(size=(3, 3)) + 3 * np.eye(3)
    Mi = np.zeros((3, 3))
    L.rb_hostmath_mat3_inv(_p(M), _p(Mi))
    assert np.allclose(Mi, np.linalg.inv(M), rtol=1e-12)


def test_synthetic_stream_is_deterministic():
    from rebvo_b200 import synth
    a = synth.Sequence(w=160, h=120, seed=3).frame(5)[1]
    b = synth.Sequence(w=160, h=120, seed=3).frame(5)[1]
    assert np.array_equal(a, b) and a.dtype == np.uint8 and a.shape == (120, 160, 3)
    c = synth.Sequence(w=160, h=120, seed=4).frame(5)[1]
    assert not np.array_equal(a, c)


def test_bias_correct_against_reference(built):
    """edge_tracker::BiasCorrect (gyro-prior fusion, SURVEY.md 8(a) K13) is pure host algebra: rb_bias_correct must
    reproduce the reference bit for bit."""
    from rebvo_b200 import capi
    from oracle import refapi
    if not refapi.available():
        pytest.skip("oracle/_ref not built")
    L, R = capi.lib(), refapi.lib()
    rng = np.random.default_rng(4)
    for _ in range(10):
        J = rng.normal(size=(30, 6))
        Wx = J.T @ J + np.eye(6)
        X = rng.normal(size=6) * 1e-2
        Gb = rng.normal(size=3) * 1e-3
        A = rng.normal(size=(3, 3))
        Wb = A @ A.T + np.eye(3) * 10
        Rg = np.eye(3) * 1e-4 + 1e-6 * (A @ A.T)
        Rb = np.eye(3) * 1e-8
        a = [np.ascontiguousarray(v.copy()) for v in (X, Wx, Gb, Wb)]
        b = [np.ascontiguousarray(v.copy()) for v in (X, Wx, Gb, Wb)]
        Rg, Rb = np.ascontiguousarray(Rg), np.ascontiguousarray(Rb)
        assert L.rb_bias_correct(_p(a[0]), _p(a[1]), _p(a[2]), _p(a[3]), _p(Rg), _p(Rb)) == 0
        R.ref_bias_correct(_p(b[0]), _p(b[1]), _p(b[2]), _p(b[3]), _p(Rg), _p(Rb))
        for x, y in zip(a, b):   # same operations in the same order (TooN's pivoting determinant included): bitwise
            assert np.array_equal(x, y)


def test_shim_imu_mirrors_compile():
    """The IMU-mode mirrors of the C++ shim (Minimizer_V, ExtRotVel, BiasCorrect) are header-only templates that the
    replay driver does not instantiate: compile them against the reference's own TooN / cam_model headers."""
    import shutil
    import subprocess
    from oracle import build_ref
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ref = build_ref.REF
    out = os.path.join(repo, "oracle", "_ref")
    if not os.path.isdir(ref) or not os.path.isdir(os.path.join(out, "toon")) or shutil.which("g++") is None:
        pytest.skip("reference headers not available here")
    cmd = ["g++", "-std=c++11", "-O0", "-w", "-fsyntax-only", "-include", os.path.join(out, "shim", "fix_gcc13.h"),
           "-I" + os.path.join(out, "shim"), "-I" + os.path.join(repo, "include"), "-I" + os.path.join(ref, "include"),
           "-I" + os.path.join(out, "toon"), os.path.join(repo, "tests", "shim_syntax.cpp")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]

