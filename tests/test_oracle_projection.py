"""oracle projection matchers == the reference's own ORBMatcher::SearchByProjection (src/ORBMatcher.cpp:51-251) and
CamModelGeneral::TransformRaysToCubemap (src/CamModelGeneral.cpp:95-154) compiled in oracle/_ref/libref.so, on reference Frame / MapPoint objects.
The reference's results are read from tests/golden/ref_oracle_projection.npz (tests/refgold.py)."""
import numpy as np
import pytest

from cubemapslam_b200 import config, synth
from oracle import ref
from tests.refgold import RECORD, gold  # noqa: F401


@pytest.fixture(scope="module")
def cam(oracle):
    cfg = config.front_1024()
    cp = oracle.cam_params(cfg)
    return cp, (ref.Ref(cp) if RECORD else None)


def test_ray_to_cubemap(oracle, cam, gold):
    cp, r = cam
    rng = np.random.default_rng(0)
    xyz = rng.normal(0, 1, (4000, 3)).astype(np.float32)
    xyz[::7, 2] = np.abs(xyz[::7, 0])                   # exactly on a face boundary (|x/z| == 1)
    xyz[::11] = 0
    uv, f = oracle.ray_to_cubemap(xyz, 650, 650)
    assert gold.same("ray_to_cubemap", (f, uv), lambda: r.ray_to_cubemap(xyz)[::-1])
    assert len(set(f.tolist())) == 6


@pytest.mark.parametrize("seed,th,ori", [(0, 15.0, True), (1, 7.0, True), (2, 15.0, False), (3, 30.0, True)])
def test_search_by_projection_last_frame(oracle, cam, gold, seed, th, ori):
    cp, r = cam
    s = synth.tracking_pair(seed, n=1500, faceW=650)
    g = oracle.FrameGrid(s["kCur"], 650, 650)
    n1, m1 = g.search_by_projection_last(s["dCur"], s["TcwCur"], s["scale"], s["kLast"], s["hasMP"], s["Xw"], s["dLast"], s["mpObs"], s["curTaken"], gold.value("cos_fov_th", lambda: r.cos_fov_th()), th, ori)
    n2, m2 = gold.value("last_%d" % seed, lambda: r.search_by_projection_last(s["kCur"], s["dCur"], s["TcwCur"], s["kLast"], s["TcwLast"], s["hasMP"], s["Xw"], s["dLast"],
                                                                          s["mpObs"], s["curTaken"], th, ori))
    m2 = np.where(m2 == -2, -1, m2)
    assert n1 == n2 and n1 > 300
    assert np.array_equal(m1, m2)
    good = m1 >= 0
    assert (s["src"][good] == m1[good]).mean() > 0.9    # and the matches are the planted correspondences


@pytest.mark.parametrize("seed,th,nn", [(0, 1.0, 0.8), (1, 3.0, 0.8), (2, 5.0, 0.6)])
def test_search_by_projection_local_map(oracle, cam, gold, seed, th, nn):
    cp, r = cam
    s = synth.tracking_pair(10 + seed, n=1500, faceW=650)
    rng = np.random.default_rng(seed)
    # the local-map variant consumes what Frame::isInFrustum stored in each MapPoint: projection, predicted level, viewing cosine
    has = s["src"] >= 0
    nMP = 1200
    pick = rng.choice(np.nonzero(has)[0], nMP, replace=False)
    proj = np.stack([s["kCur"]["x"][pick], s["kCur"]["y"][pick]], 1).astype(np.float32) + rng.normal(0, 2.0, (nMP, 2)).astype(np.float32)
    lvl = np.clip(s["kCur"]["octave"][pick] + rng.integers(0, 2, nMP), 0, 7).astype(np.int32)
    vcos = rng.choice(np.array([0.9999, 0.99, 0.7], np.float32), nMP)
    dMP = s["dLast"][s["src"][pick]]
    inView = (rng.random(nMP) < 0.9).astype(np.uint8); obs = (rng.random(nMP) < 0.9).astype(np.int32)
    taken = (rng.random(len(s["kCur"])) < 0.05).astype(np.uint8)
    g = oracle.FrameGrid(s["kCur"], 650, 650)
    n1, m1 = g.search_by_projection_local(s["dCur"], s["scale"], inView, proj, lvl, vcos, dMP, obs, taken, th, nn)
    n2, m2 = gold.value("local_%d" % seed, lambda: r.search_by_projection_local(s["kCur"], s["dCur"], inView, proj, lvl, vcos, dMP, obs, taken, th, nn))
    m2 = np.where(m2 == -2, -1, m2)
    assert n1 == n2 and n1 > 200
    assert np.array_equal(m1, m2)
