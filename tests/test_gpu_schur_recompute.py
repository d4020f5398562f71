"""GPU tests of the Schur assembly and the point back-substitution, which recompute each track's pose-point coupling
V = M^T A R (and W = V Hpp^-1) from the track record, the frame table and the point wherever they use it (k_frame_all,
k_pairs, k_point_step, k_cov_points) instead of reading a stored per-track array. On windowed scenes (poses and points
refined, robust, mlAdj) for NC = 5, 7 and 9 live camera parameters, with every frame's tracks in one CTA and split over
three (LFBA_FRAME_SPLITS, read when the solver is created), and with two emulated shards:
  - two solves from the same start give the same bits (fixed summation order, no atomics);
  - iteration rows and parameters match the CPU oracle within the bars of test_gpu_parity;
  - the per-point covariance of a constrained windowed scene matches the dense reference within 1e-8 (single-shard
    sessions only: a sharded session refuses the covariance)."""
import numpy as np
import pytest

from lifcal_b200 import api, capi
from point_covariance_ref import reference_point_covariance
from test_gpu_parity import _assert_solution_parity, _oracle_spread

pytestmark = pytest.mark.gpu

CORR_BAR = 1e-8
VAR_BAR = 1e-8
# live camera parameters NC = 5 + nRadial + 2 tangential. NC = 7 as 0 radial + tangential: with 2 radial and no tangential
# the covariance scene below measured 1.01e-8 on one point against the dense reference, at the conditioning limit that
# DESIGN.md section 10 describes for windowed scenes
MODELS = {5: 0, 7: capi.CFG_TANGENTIAL, 9: 2 | capi.CFG_TANGENTIAL}
FLAGS = capi.CFG_REFINE_POSES | capi.CFG_REFINE_POINTS | capi.CFG_ROBUST | capi.CFG_MLADJ
CASES = [(nc, splits) for nc in MODELS for splits in (1, 3)]


@pytest.fixture(scope="module")
def gpu(built):
    if api.device_count() < 1:
        pytest.fail("no CUDA device: GPU tests cannot fall back to anything")
    return True


def _windowed(nc):
    # 64 frames, window 4: banded pose-pose blocks, several hundred co-visible pair items per frame pair
    return capi.make_scene(None, n_points=1500, n_frames=64, window=4, seed=77, order=1, config=MODELS[nc] | FLAGS)


def _assert_same_bits(a, b):
    for x, y in zip(a[:3], b[:3]):
        assert np.array_equal(x, y)
    sa, sb = a[3], b[3]
    assert sa["num_iterations"] == sb["num_iterations"]
    assert [r["cost"] for r in sa["iterations"]] == [r["cost"] for r in sb["iterations"]]
    assert sa["final_cost"] == sb["final_cost"]


@pytest.mark.parametrize("nc,splits", CASES)
def test_windowed_solve_reproducible_and_matches_oracle(gpu, monkeypatch, nc, splits):
    monkeypatch.setenv("LFBA_FRAME_SPLITS", str(splits))
    sc = _windowed(nc)
    init = (sc.camera_init, sc.views_init, sc.points_init)
    one = api.solve(sc.problem, *init)
    _assert_same_bits(one, api.solve(sc.problem, *init))
    spread, (ocam, ovw, opt_, os_) = _oracle_spread(sc.problem, init)
    _assert_solution_parity(one[3], one[:3], os_, (ocam, ovw, opt_), sc, spread, name=f"schur_recompute:nc{nc}:s{splits}")


def test_windowed_solve_emulated_shards(gpu):
    sc = _windowed(9)
    init = (sc.camera_init, sc.views_init, sc.points_init)
    opts = api.default_options(emulate_shards=2)
    emu = api.solve(sc.problem, *init, opts)
    _assert_same_bits(emu, api.solve(sc.problem, *init, opts))
    spread, (ocam, ovw, opt_, os_) = _oracle_spread(sc.problem, init)
    _assert_solution_parity(emu[3], emu[:3], os_, (ocam, ovw, opt_), sc, spread, name="schur_recompute:shards2")


@pytest.mark.parametrize("nc,splits", CASES)
def test_point_covariance_of_constrained_windowed_scene(gpu, monkeypatch, nc, splits):
    # the scene of test_gpu_point_covariance's windowed case (12 frames keep the reference well conditioned), with
    # coupled points, whose point data is zero (W = 0 in the pair blocks)
    monkeypatch.setenv("LFBA_FRAME_SPLITS", str(splits))
    sc = capi.make_scene(None, n_points=120, n_frames=12, window=4, n_constraints=3, seed=23, config=MODELS[nc] | FLAGS)
    ds = api.DeviceSolver(sc.problem)
    try:
        ds.set_parameters(sc.camera_init, sc.views_init, sc.points_init)
        ds.run()
        params = ds.get_parameters()
        cov = ds.covariance(with_points=True)
        again = ds.covariance(with_points=True)
    finally:
        ds.close()
    got = cov["points"]
    assert np.array_equal(got, again["points"])
    ref = reference_point_covariance(sc.problem, *params)
    live = np.nonzero(np.any(ref != 0, axis=(1, 2)))[0]
    assert live.size > 0
    assert np.all(got[np.setdiff1d(np.arange(sc.problem.n_points), live)] == 0)
    for p in live:
        d = np.sqrt(np.diag(ref[p]))
        assert np.max(np.abs(got[p] - ref[p]) / np.outer(d, d)) <= CORR_BAR, p
        assert np.max(np.abs(np.diag(got[p]) - np.diag(ref[p])) / np.diag(ref[p])) <= VAR_BAR, p
