"""Plain references and problem builders for the device tracking chain (frame index -> SearchByProjection(last frame) -> pose-input gather ->
PoseOptimization). numpy only; the GPU tests in test_gpu_tracking_chain.py and the CPU checks in test_oracle_tracking_chain.py share them."""
import functools

import numpy as np

from cubemapslam_b200 import synth

KP_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"), ("octave", "<i4"), ("class_id", "<i4")])


def scale_factors(nlevels=8, factor=1.2):
    sc = np.ones(nlevels, np.float32)
    for l in range(1, nlevels):
        sc[l] = sc[l - 1] * np.float32(factor)
    return sc


def inv_sigma2_levels(nlevels=8, factor=1.2):
    sc = scale_factors(nlevels, factor)
    return (np.float32(1.0) / (sc * sc)).astype(np.float32)


def cos_fov_th(fov_deg):
    """CamModelGeneral::SetCosFovTh (reference include/CamModelGeneral.h:224-229): float argument, double cos, float result."""
    a = np.float32(fov_deg) / np.float32(2) * (np.float32(3.1415926535897932384626) / np.float32(180))
    return np.float32(np.cos(np.float64(a)))


def gather_ref(match, kCur, nCur, stride, rays, cth, XwLast, inv_sigma2_levels):
    """What Tracking hands PoseOptimization (reference src/Optimizer.cpp:80-131): the matched slots of the current frame, in slot order.

    match: current-frame slot -> LastFrame index (-1: none, -2: assigned, then cleared by the rotation check), kCur: the frame's key points,
    nCur: its key-point count (clamped to `stride`, the row length of match / kCur / rays). A slot is kept iff match >= 0 and not
    ray.z < cth (src/Optimizer.cpp:82-84; a NaN z and z == cth are kept); rays=None keeps every matched slot. The weight is
    inv_sigma2[octave]. Returns (Xw (count, 3), kp (count, 2), w (count,)) float32 and count."""
    n = min(int(nCur), int(stride))
    m = np.asarray(match[:n], np.int64)
    keep = m >= 0
    if rays is not None:
        z = np.asarray(rays, np.float32).reshape(-1, 3)[:n, 2]
        keep &= ~(z < np.float32(cth))
    slots = np.nonzero(keep)[0]
    k = np.asarray(kCur)[slots]
    Xw = np.asarray(XwLast, np.float32).reshape(-1, 3)[m[slots]]
    kp = np.stack([k["x"], k["y"]], 1).astype(np.float32).reshape(-1, 2)
    w = np.asarray(inv_sigma2_levels, np.float32)[k["octave"]]
    return Xw, kp, w, len(slots)


def perturb_pose(T, rot, trans, rng):
    """T (4x4) with its rotation turned by a random axis-angle of norm `rot` (rad) and its translation moved by a random vector of norm `trans`."""
    def unit():
        v = rng.normal(size=3)
        return v / np.linalg.norm(v)
    T = np.asarray(T, np.float64)
    out = np.eye(4)
    out[:3, :3] = synth._rodrigues(rot * unit()) @ T[:3, :3]
    out[:3, 3] = T[:3, 3] + trans * unit()
    return out.astype(np.float32)


@functools.lru_cache(maxsize=None)
def _pose_base(faceW, seed, outlier_frac):
    return synth.pose_problem(n=4096, faceW=faceW, seed=seed, outlier_frac=outlier_frac)


def pose_case(n, faceW=650, seed=0, outlier_frac=0.15, offset=0, rot=None, trans=None):
    """A PoseOptimization frame of exactly n correspondences (n <= 4096): the edges [offset, offset + n) of a 4096-edge synth.pose_problem
    (points all around the camera, so every cube face is observed; `outlier_frac` of the observations carry +-30 px of extra noise).
    The prior is pose_problem's (1e-2 per rotation / translation component) unless rot / trans (rad, world units) ask for another one."""
    b = _pose_base(int(faceW), int(seed), float(outlier_frac))
    assert n + offset <= len(b["Xw"]), (n, offset, len(b["Xw"]))
    sl = slice(offset, offset + n)
    T = b["Tcw"].copy()
    if rot is not None or trans is not None:
        T = perturb_pose(b["Tcw_true"], rot or 0.0, trans or 0.0, np.random.default_rng(1000 + seed + 7 * n + offset))
    return dict(Tcw=T, Xw=b["Xw"][sl].copy(), kpxy=b["kpxy"][sl].copy(), inv_sigma2=b["inv_sigma2"][sl].copy(), faceW=faceW, Tcw_true=b["Tcw_true"])


def plant_observation(q, i, dx):
    """q with observation i moved to its exact projection under the planted pose plus dx pixels in x, at octave-0 weight 1 (chi2 ~ dx^2)."""
    W = q["faceW"]
    T = np.asarray(q["Tcw_true"], np.float64)
    Xc = T[:3, :3] @ q["Xw"][i].astype(np.float64) + T[:3, 3]
    u, v = synth._rays_to_cubemap(Xc[0], Xc[1], Xc[2], W)
    q = dict(q, kpxy=q["kpxy"].copy(), inv_sigma2=q["inv_sigma2"].copy())
    q["kpxy"][i] = (u + dx, v); q["inv_sigma2"][i] = 1.0
    return q


def tracking_task(seed, n=3000, faceW=650, rot=0.004, trans=0.01, angle_frac=0.15):
    """A SearchByProjection(last frame) + PoseOptimization task on synth.tracking_pair: the planted TcwCur is kept as the truth and the prior
    ("Tcw") is it perturbed by `rot` rad / `trans`. The angles of `angle_frac` of the current key points are redrawn, so the rotation check
    clears some assigned slots to -2 (the pair as generated produces almost none)."""
    s = synth.tracking_pair(seed, n=n, faceW=faceW)
    rng = np.random.default_rng(5000 + seed)
    k = s["kCur"].copy()
    pick = rng.random(len(k)) < angle_frac
    k["angle"][pick] = rng.uniform(0, 360, int(pick.sum())).astype(np.float32)
    s["kCur"] = k
    s["Ttrue"] = s["TcwCur"].copy()
    s["Tcw"] = perturb_pose(s["TcwCur"], rot, trans, rng)
    return s


def oracle_chain(orc, s, cth, th=15.0, check_ori=True):
    """The CPU chain on one task: FrameGrid.search_by_projection_last -> gather_ref -> oracle.pose_opt (prior s["Tcw"])."""
    W = s["faceW"]
    g = orc.FrameGrid(s["kCur"], W, W)
    nm, match = g.search_by_projection_last(s["dCur"], s["Tcw"], s["scale"], s["kLast"], s["hasMP"], s["Xw"], s["dLast"], s["mpObs"], s["curTaken"], cth, th, check_ori)
    rays, _ = orc.key_point_rays(s["kCur"], W, W)
    Xw, kp, w, cnt = gather_ref(match, s["kCur"], len(s["kCur"]), len(s["kCur"]), rays, cth, s["Xw"], inv_sigma2_levels())
    po = orc.pose_opt(s["Tcw"], Xw, kp, w, W, W)
    return dict(nmatches=nm, match=match, rays=rays, Xw=Xw, kp=kp, w=w, count=cnt, pose=po)


def pose_errors(T, Ttrue):
    """(rotation angle in rad, translation distance) between two Tcw."""
    T = np.asarray(T, np.float64); Ttrue = np.asarray(Ttrue, np.float64)
    dR = T[:3, :3] @ Ttrue[:3, :3].T
    ang = float(np.arccos(np.clip((np.trace(dR) - 1) / 2, -1, 1)))
    return ang, float(np.linalg.norm(T[:3, 3] - Ttrue[:3, 3]))
