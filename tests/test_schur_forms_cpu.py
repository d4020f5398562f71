"""CPU test of the camera-frame Schur helpers in lifcal_b200/csrc/lfba_math.cuh (the functions k_points, k_frame_all,
k_pairs, k_point_step and k_cov_points call), compiled for the host by tests/cpu_harness/schur_forms.cpp: the pose
block, pose gradient, camera-pose block, frame-pair block and point back substitution built with the point eliminated
inside the 3 x 3 camera-frame block equal the same terms written through V = M^T A R and W = V Hpp^-1."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
BAR = 1e-13


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    src = os.path.join(HERE, "cpu_harness", "schur_forms.cpp")
    out = str(tmp_path_factory.mktemp("schur_forms") / "libschur_forms.so")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.check_call([cxx, "-O2", "-fPIC", "-std=c++17", "-shared", "-x", "c++", "-o", out, src])
    L = C.CDLL(out)
    dp = C.POINTER(C.c_double)
    L.schur_forms.argtypes = [C.c_int] + [dp] * 15
    L.track_w_forms.argtypes = [dp] * 6
    return L


def _p(a):
    return np.ascontiguousarray(a, dtype=np.float64).ctypes.data_as(C.POINTER(C.c_double))


def _upper(S):
    return np.array([S[0, 0], S[0, 1], S[0, 2], S[1, 1], S[1, 2], S[2, 2]])


def _spd(rng, scale):
    G = rng.standard_normal((5, 3))
    return scale * (G.T @ G / 5 + 0.5 * np.eye(3))


def _frame(rng):
    fe = np.zeros(40)
    q, _ = np.linalg.qr(rng.standard_normal((3, 3)))
    fe[0:9] = q.ravel()
    fe[9:36] = rng.standard_normal(27)  # dR/da_k: any 3 x 3 for the identity
    fe[36:39] = rng.standard_normal(3)
    return fe


def _rel(a, b):
    return np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300)


@pytest.mark.parametrize("nc", [5, 6, 7, 8, 9])
def test_camera_frame_schur_terms_match_vw_form(lib, nc):
    rng = np.random.default_rng(100 + nc)
    worst = 0.0
    for _ in range(50):
        A1, A2 = _upper(_spd(rng, 10.0)), _upper(_spd(rng, 10.0))
        b1 = rng.standard_normal(3)
        C1 = rng.standard_normal((3, nc))
        fe1, fe2 = _frame(rng), _frame(rng)
        X = rng.standard_normal(3) * 2 + np.array([0, 0, 5.0])
        Hi = _upper(np.linalg.inv(_spd(rng, 20.0)))
        gp = rng.standard_normal(3)
        Hcp = rng.standard_normal((nc, 3))
        y1, y2, yc = rng.standard_normal(6), rng.standard_normal(6), rng.standard_normal(nc)
        n = 21 + 6 + 6 * nc + 36 + 3
        ref, fac = np.zeros(n), np.zeros(n)
        lib.schur_forms(nc, _p(A1), _p(b1), _p(C1), _p(fe1), _p(A2), _p(fe2), _p(X), _p(Hi), _p(gp), _p(Hcp),
                        _p(y1), _p(y2), _p(yc), _p(ref), _p(fac))
        o = np.cumsum([0, 21, 6, 6 * nc, 36, 3])
        for name, a, b in zip(["S_ff", "g_f", "S_cf", "S_f1f2", "y_p"], o[:-1], o[1:]):
            r = _rel(fac[a:b], ref[a:b])
            assert r < BAR, (name, r)
            worst = max(worst, r)
        w_ref, w_fac = np.zeros(18), np.zeros(18)
        lib.track_w_forms(_p(A1), _p(fe1), _p(X), _p(Hi), _p(w_ref), _p(w_fac))
        assert _rel(w_fac, w_ref) < BAR
    assert worst > 0.0  # the two forms round differently: the comparison is not vacuous
