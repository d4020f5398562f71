"""CPU tests of the step before the solve (SURVEY.md 8(f) N2): the oracle's restatement of the epipolar web and of
projectPointsToRawImage (oracle/project_raw.hpp), and the product's host-side web (lfba_epipolar_web)."""
import ctypes as C

import numpy as np
import pytest

import helpers
from lifcal_b200 import api
from oracle import binding as ob


def test_epipolar_primitives_equal_the_reference_class_bit_for_bit(built):
    R = ob.ref_lib()
    if R is None or not hasattr(R, "ref_epi_make"):
        pytest.skip("oracle/_ref not built: needs the upstream LiFCal sources (make -C oracle ref REF=<LiFCal checkout>)")
    L = ob.lib()
    rng = np.random.default_rng(5)
    a, b, o, r = (np.zeros(3) for _ in range(4))
    dp = lambda v: v.ctypes.data_as(C.POINTER(C.c_double))
    for k in range(2000):
        x, y, d = rng.normal(), rng.normal(), 23.0 * (1 + rng.random() * 9)
        if k % 50 == 0:
            x, y = 1.0, 0.0  # the "already unit length" branch (squared length == 1.0f)
        L.oracle_epi_make(x, y, d, dp(o))
        R.ref_epi_make(x, y, d, dp(r))
        assert np.array_equal(o, r)
        a[:] = o
        L.oracle_epi_make(rng.normal(), rng.normal(), 23.0, dp(b))
        L.oracle_epi_add(dp(a), dp(b), dp(o))
        R.ref_epi_add(dp(a), dp(b), dp(r))
        assert np.array_equal(o, r)


@pytest.mark.parametrize("D,rot,on", [(23.0, 0.003, True), (23.0, 0.0, False), (34.5, -0.01, True), (14.0, 0.02, True)])
def test_web_structure_and_product_host_web_equals_oracle(built, D, rot, on):
    lines, gb = ob.epi_web(D, rot, on)
    pl, pg = api.epipolar_web(D, rot, on)
    assert np.array_equal(lines, pl) and np.array_equal(gb, pg)  # two independent restatements, same bits
    dist = lines[:, 2]
    first = dist[gb[:-1]]
    assert np.all(np.diff(first) > 0)                       # groups ascending by base-line length
    assert np.all(dist <= np.float32(D) * 10 + 1e-9)        # maxDist = 10 lens diameters
    assert np.allclose(np.hypot(lines[:, 0], lines[:, 1]), 1.0, atol=1e-12)
    assert np.all(lines[:, 1] > -1.0)                       # lines against the y unit vector are dropped
    for g0, g1 in zip(gb[:-1], gb[1:]):                     # float-equal length inside a group
        assert np.all(np.float32(dist[g0:g1]) == np.float32(dist[g0]))
    # the web is half of the hexagonal lattice within 10 D (each line stands for +/- direction)
    assert abs(2 * len(lines) - np.pi * 100 / np.sqrt(0.75)) < 40
    # every line is a lattice vector i e0 + j e1 of the (rotated) hexagonal lattice
    e0 = lines[np.argmin(np.abs(lines[:, 1] - (-np.sin(rot) if on else 0)) + np.abs(dist - D))]
    v = lines[:, :2] * dist[:, None]
    ca, sa = (np.cos(np.float32(rot)), np.sin(np.float32(rot))) if on else (1.0, 0.0)
    u = np.stack([v[:, 0] * ca - v[:, 1] * sa, v[:, 0] * sa + v[:, 1] * ca], 1) / np.float32(D)  # back-rotated, in units of D
    j = u[:, 1] / np.sqrt(0.75)
    i = u[:, 0] - 0.5 * j
    assert np.allclose(j, np.round(j), atol=1e-6) and np.allclose(i, np.round(i), atol=1e-6)


def test_projection_oracle_geometry(built):
    g = helpers.make_lens_grid(raw=512)
    rng = np.random.default_rng(11)
    m = 3000
    fx = rng.random(m) * (512 / 2 - 1)
    fy = rng.random(m) * (512 / 2 - 1)
    vd = 1.5 + rng.random(m) * 20
    o = ob.project_to_raw(g, fx, fy, vd)
    assert o["obs_x"].size > 10 * m * 0.5
    f = o["feature"]
    v = np.float32(vd)[f]
    assert np.all((v > 2.0) & (v < 20.0))                    # :655
    xu = np.float32(2) * (np.float32(fx) + np.float32(0.5)) - np.float32(0.5)
    yu = np.float32(2) * (np.float32(fy) + np.float32(0.5)) - np.float32(0.5)
    cx, cy = np.float32(o["ml_x"]), np.float32(o["ml_y"])
    assert np.array_equal(cx.astype(np.float64), o["ml_x"])  # float32 values widened (MicroLens.h:22-23)
    assert np.array_equal(np.float32(o["obs_x"]).astype(np.float64), o["obs_x"])
    # micro-image relation x_R = c + (x_V - c) / v  (:748-749), float32-exact
    assert np.array_equal(np.float32(o["obs_x"]), (xu[f] - cx) / v + cx)
    assert np.array_equal(np.float32(o["obs_y"]), (yu[f] - cy) / v + cy)
    # inside the valid part of the micro image (:759) and inside the search radius D/2 v + 2 (:661)
    r2 = (np.float32(o["obs_x"]) - cx) ** 2 + (np.float32(o["obs_y"]) - cy) ** 2
    assert np.all(r2 < g.lens_validity_radius_2)
    rad = g.lens_diameter * np.float32(0.5) * v + np.float32(2)
    assert np.all((cx - xu[f]) ** 2 + (cy - yu[f]) ** 2 <= rad * rad * (1 + 1e-6))
    # completeness: every lens well inside the radius whose micro image holds a valid point is found, none twice
    k = 17
    sel = f == f[np.searchsorted(f, f[k])]
    feat = f[k]
    found = set(zip(cx[f == feat].tolist(), cy[f == feat].tolist()))
    # (reference behaviour, mirrored: a lens can be visited twice — predicted centres outside the image are clamped onto
    #  border pixels (:729-732), and a ROTATED grid's web holds pairs of exactly opposite lines because only the direction
    #  (0, -1) is filtered (:599))
    d2 = (g.lens_cx - xu[feat]) ** 2 + (g.lens_cy - yu[feat]) ** 2
    radk = float(g.lens_diameter) * 0.5 * float(np.float32(vd[feat])) + 2.0
    for l in np.where(d2 < (radk - 1.5) ** 2)[0]:
        xr = (xu[feat] - g.lens_cx[l]) / np.float32(vd[feat]) + g.lens_cx[l]
        yr = (yu[feat] - g.lens_cy[l]) / np.float32(vd[feat]) + g.lens_cy[l]
        inside = 0 <= xr <= 511 and 0 <= yr <= 511 and (xr - g.lens_cx[l]) ** 2 + (yr - g.lens_cy[l]) ** 2 < g.lens_validity_radius_2 * 0.98
        centre_px_valid = 0 <= g.lens_cx[l] <= 511 and 0 <= g.lens_cy[l] <= 511
        if inside and centre_px_valid:
            assert (float(g.lens_cx[l]), float(g.lens_cy[l])) in found
    assert sel.any()
    # frame-major order is preserved: feature indices ascend
    assert np.all(np.diff(f) >= 0)
    # an unrotated grid has no opposite lines: away from the image border every lens is visited at most once per feature
    g0 = helpers.make_lens_grid(raw=512, rotation=0.0)
    g0.rotation_on_grid = 0
    vi = 2.5 + rng.random(300) * 4
    o0 = ob.project_to_raw(g0, 90 + rng.random(300) * 70, 90 + rng.random(300) * 70, vi)
    key = np.stack([o0["feature"].astype(np.float64), o0["ml_x"], o0["ml_y"]], 1)
    assert len(key) > 3000 and len(np.unique(key, axis=0)) == len(key)
