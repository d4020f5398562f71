"""CPU tests (no GPU): the oracle's restated functor against
  (a) the committed golden vectors made by the REFERENCE's own headers (tests/golden/functor_kat.npz),
  (b) the reference functors live, when oracle/_ref/libref_functor.so is present,
  (c) central finite differences (sanity of the autodiff restatement).
Reference: src/BundleAdjustment/BundleAdjustment.h:120-195,262-267; src/CameraModel.h:87-264."""
import ctypes as C
import os

import numpy as np
import pytest

import helpers
from lifcal_b200 import capi
from oracle import binding as ob

GOLD = os.path.join(os.path.dirname(__file__), "golden", "functor_kat.npz")
NO_REF = "oracle/_ref not built: needs the upstream LiFCal sources (make -C oracle ref REF=<LiFCal checkout>)"
ARITY_BITS = [capi.CFG_REFINE_POSES | capi.CFG_REFINE_POINTS, capi.CFG_REFINE_POSES, 0]


def _problem(cfg, spx, scale, obs, ml):
    n = obs.shape[0]
    return capi.ProblemArrays(cfg, 0, spx, spx, scale, n, n, obs[:, 0], obs[:, 1], ml[:, 0], ml[:, 1],
                              np.arange(n), np.arange(n))


def _relerr(a, b):
    return np.max(np.abs(a - b) / (1e-300 + np.maximum(np.abs(a), np.abs(b)) + 1e-9 * np.max(np.abs(b))))


def test_oracle_matches_reference_golden(built):
    g = np.load(GOLD)
    spx, scale = float(g["spx"][0]), float(g["scale"][0])
    checked = 0
    for mc in helpers.all_model_configs():
        for ab in ARITY_BITS:
            cfg = mc | ab
            for ci in range(2):
                key = f"cfg{cfg:#06x}_{ci}"
                pa = _problem(cfg, spx, scale, g[key + "_obs"], g[key + "_ml"])
                ev = ob.evaluate(pa, g[key + "_camera"], g[key + "_views"].ravel(), g[key + "_points"].ravel())
                # residuals: absolute 1e-9 px is far below the 1e-9 relative bar on |r| ~ px
                assert np.max(np.abs(ev["residuals"] - g[key + "_res"])) < 1e-9, key
                assert _relerr(ev["jac_camera"], g[key + "_jc"]) < 1e-10, key
                assert _relerr(ev["jac_view"], g[key + "_jv"]) < 1e-10, key
                assert _relerr(ev["jac_point"], g[key + "_jp"]) < 1e-10, key
                checked += 1
    assert checked == 12 * 3 * 2


@pytest.mark.skipif(ob.ref_lib() is None, reason=NO_REF)
def test_oracle_matches_reference_live(built):
    rng = np.random.default_rng(7)
    worst = 0.0
    for mc in helpers.all_model_configs():
        for ab in ARITY_BITS:
            cfg = mc | ab
            b = helpers.random_blocks(rng, cfg, 64, signs=True)
            pa = _problem(cfg, b["spx"], b["scale"], b["obs"], b["ml"])
            a = ob.evaluate(pa, b["cams"][0], b["views"].ravel(), b["points"].ravel())
            r = ob.evaluate(pa, b["cams"][0], b["views"].ravel(), b["points"].ravel(), use_ref=True)
            assert np.max(np.abs(a["residuals"] - r["residuals"])) < 1e-10
            for k in ("jac_camera", "jac_view", "jac_point"):
                e = _relerr(a[k], r[k])
                worst = max(worst, e)
                assert e < 1e-11, (hex(cfg), k, e)
            assert abs(a["cost"] - r["cost"]) <= 1e-12 * abs(r["cost"])
    print("worst relative Jacobian difference oracle vs reference:", worst)


def test_distance_constraint_golden(built):
    g = np.load(GOLD)
    # the oracle evaluates constraints inside solve/eval cost; check the value through a 2-point problem cost
    p1, p2, dist, sig, res = g["dc_p1"], g["dc_p2"], g["dc_dist"], g["dc_sigma"], g["dc_res"]
    for i in range(p1.shape[0]):
        pts = np.concatenate([p1[i], p2[i]])
        cfg = capi.CFG_REFINE_POSES | capi.CFG_REFINE_POINTS
        pa = capi.ProblemArrays(cfg, 0, 0.011, 0.011, 2.0, 1, 2, np.zeros(0), np.zeros(0), np.zeros(0), np.zeros(0),
                                np.zeros(0, np.int32), np.zeros(0, np.int32), [0], [1], [dist[i]], [sig[i]])
        cam = np.zeros(17)
        cam[:5] = [35, 33, 0.5, 500, 500]
        ev = ob.evaluate(pa, cam, np.zeros(6), pts, jacobians=False)
        assert abs(ev["cost"] - 0.5 * res[i] ** 2) <= 1e-12 * max(1.0, 0.5 * res[i] ** 2)


def test_oracle_jacobian_vs_finite_differences(built):
    rng = np.random.default_rng(3)
    cfg = 2 | capi.CFG_TANGENTIAL | capi.CFG_MLADJ | capi.CFG_REFINE_POSES | capi.CFG_REFINE_POINTS
    b = helpers.random_blocks(rng, cfg, 16)
    pa = _problem(cfg, b["spx"], b["scale"], b["obs"], b["ml"])
    cam, vw, pt = b["cams"][0], b["views"].ravel().copy(), b["points"].ravel().copy()
    ev = ob.evaluate(pa, cam, vw, pt)

    def res(c, v, p):
        return ob.evaluate(pa, c, v, p, jacobians=False)["residuals"]

    for j in range(9):
        h = 1e-6 * max(1e-3, abs(cam[j]))
        cp, cm = cam.copy(), cam.copy()
        cp[j] += h
        cm[j] -= h
        fd = (res(cp, vw, pt) - res(cm, vw, pt)) / (2 * h)
        an = ev["jac_camera"][:, :, j]
        assert np.max(np.abs(fd - an)) <= 2e-5 * (1 + np.max(np.abs(an))), j
    for j in range(6):
        h = 1e-6 if j < 3 else 1e-4
        vp, vm = vw.copy().reshape(-1, 6), vw.copy().reshape(-1, 6)
        vp[:, j] += h
        vm[:, j] -= h
        fd = (res(cam, vp.ravel(), pt) - res(cam, vm.ravel(), pt)) / (2 * h)
        an = ev["jac_view"][:, :, j]
        assert np.max(np.abs(fd - an)) <= 2e-5 * (1 + np.max(np.abs(an))), j
    for j in range(3):
        h = 1e-3
        pp, pm = pt.copy().reshape(-1, 3), pt.copy().reshape(-1, 3)
        pp[:, j] += h
        pm[:, j] -= h
        fd = (res(cam, vw, pp.ravel()) - res(cam, vw, pm.ravel())) / (2 * h)
        an = ev["jac_point"][:, :, j]
        assert np.max(np.abs(fd - an)) <= 2e-5 * (1 + np.max(np.abs(an))), j


@pytest.mark.skipif(ob.ref_lib() is None, reason=NO_REF)
def test_pose_matrix_matches_reference(built):
    R = ob.ref_lib()
    rng = np.random.default_rng(5)
    for _ in range(50):
        v = np.concatenate([rng.uniform(-3, 3, 3), 100 * rng.standard_normal(3)])
        out = np.zeros(16)
        R.ref_pose_matrix(capi._dp(v), capi._dp(out))
        M = out.reshape(4, 4)
        a = v[:3]
        cx, sx, cy, sy, cz, sz = np.cos(a[0]), np.sin(a[0]), np.cos(a[1]), np.sin(a[1]), np.cos(a[2]), np.sin(a[2])
        Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
        Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
        Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
        assert np.allclose(M[:3, :3], Rx @ Ry @ Rz, atol=1e-14)
        assert np.allclose(M[:3, 3], v[3:])
        assert np.allclose(M[3], [0, 0, 0, 1])
