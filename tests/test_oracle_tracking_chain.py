"""The CPU side of the tracking-chain parity tests: gather_ref on hand-made frames, and the oracle chain (SearchByProjection(last frame) ->
gather -> PoseOptimization) on planted tasks, which must recover the planted pose better than the prior. CPU only."""
import numpy as np
import pytest

from cubemapslam_b200 import config

from . import tracking_chain_ref as R


def _kps(xy_oct):
    k = np.zeros(len(xy_oct), R.KP_DTYPE)
    for i, (x, y, o) in enumerate(xy_oct):
        k[i] = (x, y, 31, 0, 0, o, -1)
    return k


def test_gather_ref_hand_made():
    isg = R.inv_sigma2_levels()
    cth = np.float32(-0.25)
    k = _kps([(10, 11, 0), (20, 21, 3), (30, 31, 7), (40, 41, 1), (50, 51, 2), (60, 61, 5), (70, 71, 4), (80, 81, 6)])
    XwL = np.arange(30, dtype=np.float32).reshape(10, 3)
    match = np.array([3, -1, 9, -2, 0, 5, 7, 1], np.int32)
    rays = np.zeros((8, 3), np.float32); rays[:, 2] = 1
    rays[2, 2] = cth                                      # z == cth: kept
    rays[5, 2] = np.nextafter(cth, np.float32(-np.inf))   # just below: dropped
    rays[6, 2] = np.nan                                   # NaN: kept (the test is `z < cth`)
    rays[7, 2] = 0
    Xw, kp, w, n = R.gather_ref(match, k, 8, 8, rays, cth, XwL, isg)
    slots = [0, 2, 4, 6, 7]
    assert n == 5
    assert np.array_equal(Xw, XwL[match[slots]])
    assert np.array_equal(kp, np.stack([k["x"][slots], k["y"][slots]], 1))
    assert np.array_equal(w, isg[k["octave"][slots]]) and w.dtype == np.float32
    # no ray filter: the dropped slot comes back, order kept
    Xw2, _, _, n2 = R.gather_ref(match, k, 8, 8, None, cth, XwL, isg)
    assert n2 == 6 and np.array_equal(Xw2, XwL[match[[0, 2, 4, 5, 6, 7]]])
    # nCur is clamped to the stride; slots past nCur are ignored
    assert R.gather_ref(match, k, 100, 4, rays, cth, XwL, isg)[3] == 2
    assert R.gather_ref(match, k, 3, 8, rays, cth, XwL, isg)[3] == 2
    Xw0, kp0, w0, n0 = R.gather_ref(match, k, 0, 8, rays, cth, XwL, isg)
    assert n0 == 0 and Xw0.shape == (0, 3) and kp0.shape == (0, 2) and w0.shape == (0,)


def test_gather_ref_all_dropped():
    k = _kps([(1, 1, 0)] * 4)
    assert R.gather_ref(np.array([-1, -2, -1, -2], np.int32), k, 4, 4, None, 0.0, np.zeros((1, 3), np.float32), R.inv_sigma2_levels())[3] == 0


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_oracle_chain_recovers_the_planted_pose(oracle, seed):
    cth = R.cos_fov_th(config.front_1024()["Camera.fov"])
    s = R.tracking_task(seed)
    c = R.oracle_chain(oracle, s, cth)
    m = c["match"]
    assert 1000 < c["count"] <= c["nmatches"]
    assert np.all(s["src"][m >= 0] == m[m >= 0])                    # no wrong associations
    a0, t0 = R.pose_errors(s["Tcw"], s["Ttrue"])
    a1, t1 = R.pose_errors(c["pose"]["Tcw"], s["Ttrue"])
    assert t1 < 0.5 * t0 and t1 < 5e-3 and a1 < a0
    assert c["pose"]["inliers"] > 0.9 * c["count"]


def test_tracking_task_clears_slots_in_the_rotation_check(oracle):
    """The redrawn angles make the rotation histogram drop assignments: with the check on, fewer matches than with it off."""
    cth = R.cos_fov_th(config.front_1024()["Camera.fov"])
    s = R.tracking_task(0)
    g = oracle.FrameGrid(s["kCur"], 650, 650)
    args = (s["dCur"], s["Tcw"], s["scale"], s["kLast"], s["hasMP"], s["Xw"], s["dLast"], s["mpObs"], s["curTaken"], cth, 15.0)
    n_on, _ = g.search_by_projection_last(*args, True)
    n_off, _ = g.search_by_projection_last(*args, False)
    assert n_on < n_off


@pytest.mark.parametrize("n", [3, 10, 257, 4096])
def test_pose_case_sizes(n):
    p = R.pose_case(n, faceW=450, seed=1, outlier_frac=0.5, offset=0)
    assert len(p["Xw"]) == n and p["kpxy"].shape == (n, 2) and p["inv_sigma2"].shape == (n,)
    q = R.pose_case(n, rot=0.05, trans=0.02)
    a, t = R.pose_errors(q["Tcw"], q["Tcw_true"])
    assert abs(a - 0.05) < 1e-6 and abs(t - 0.02) < 1e-6


def test_plant_observation(oracle):
    q = R.pose_case(300, faceW=650, seed=1, outlier_frac=0.15, rot=0.1, trans=0.05)
    p = R.plant_observation(q, 7, 2.47428)
    err, _, _, _ = oracle.edge_eval(q["Tcw_true"], p["Xw"][7].astype(np.float64), p["kpxy"][7, 0], p["kpxy"][7, 1], 650, 650)
    assert abs(np.hypot(*err) - 2.47428) < 1e-3 and p["inv_sigma2"][7] == 1
    assert np.array_equal(np.delete(p["kpxy"], 7, 0), np.delete(q["kpxy"], 7, 0))
    # the frame of test_gpu_tracking_chain.py::test_pose_optimization_robust_switch_round
    assert oracle.pose_opt(p["Tcw"], p["Xw"], p["kpxy"], p["inv_sigma2"], 650, 650)["inliers"] == 259
