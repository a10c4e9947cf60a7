"""oracle LocalMapping feature operations (oracle/mapping.h) == the reference's own MapPoint::ComputeDistinctiveDescriptors (src/MapPoint.cpp:243-303),
ORBMatcher::Fuse (src/ORBMatcher.cpp:1126-1240), ORBMatcher::SearchForTriangulation (:971-1124) and CamModelGeneral::GetVectorSigma
(src/CamModelGeneral.cpp:307-335) compiled in oracle/_ref/libref.so, run on reference KeyFrame / MapPoint objects.
The reference's results are read from tests/golden/ref_oracle_mapping.npz (tests/refgold.py)."""
import numpy as np
import pytest

from cubemapslam_b200 import config, synth
from oracle import ref
from tests.refgold import RECORD, gold  # noqa: F401


@pytest.fixture(scope="module")
def cam(oracle):
    cp = oracle.cam_params(config.front_1024())
    return cp, (ref.Ref(cp) if RECORD else None)


def test_distinctive_descriptor(oracle, cam, gold):
    cp, r = cam
    rng = np.random.default_rng(0)
    sets = []
    for N in (1, 2, 3, 4, 7, 12, 33):
        for rep in range(6):
            base = rng.integers(0, 256, 32, dtype=np.uint8)
            d = np.stack([base ^ np.packbits(rng.random(256) < rng.uniform(0.02, 0.3), bitorder="little") for _ in range(N)])
            if rep == 0 and N > 2:
                d[1] = d[0]                                # ties: the first index with the least median wins
            sets.append(d)
    want = gold.value("distinctive", lambda: np.stack([r.distinctive_descriptor(d) for d in sets]))
    for d, w in zip(sets, want):
        best = oracle.distinctive_descriptors(d, np.array([0, len(d)], np.int32))[0]
        assert np.array_equal(w, d[best])
    assert oracle.distinctive_descriptors(np.zeros((0, 32), np.uint8), np.array([0, 0], np.int32))[0] == -1


def test_vector_sigma(oracle, cam, gold):
    cp, r = cam
    rng = np.random.default_rng(1)
    tiles = [(1, 1), (0, 1), (2, 1), (1, 0), (1, 2)]
    cases = []
    for i in range(400):
        c, rr = tiles[i % 5]
        kx = np.float32(c * 650 + rng.uniform(0, 649.9)); ky = np.float32(rr * 650 + rng.uniform(0, 649.9))
        cases.append((kx, ky, rng.normal(0, 1, 3).astype(np.float32)))
    want = gold.value("vector_sigma", lambda: np.array([r.vector_sigma(*c) for c in cases]))
    for i, (c, b) in enumerate(zip(cases, want)):
        a = oracle.vector_sigma(*c, 650, 650)
        assert a == b or (np.isnan(a) and np.isnan(b)), (i, a, b)


@pytest.mark.parametrize("seed,th", [(0, 3.0), (1, 3.0), (2, 6.0)])
def test_fuse_search(oracle, cam, gold, seed, th):
    cp, r = cam
    s = synth.mapping_pair(seed, n=1500, faceW=650)
    nf, valid, level, idx = gold.value("fuse_%d" % seed, lambda: r.fuse(s["kCur"], s["dCur"], s["TcwCur"], s["Xw"], s["kLast"], s["dLast"], s["TcwLast"], th))
    g = oracle.FrameGrid(s["kCur"], 650, 650)
    bi, bd = g.fuse_search(s["dCur"], s["TcwCur"], s["scale"], s["inv_level_sigma2"], valid, s["Xw"], level, s["dLast"], th)
    fused = bd <= 50
    assert nf == int(fused.sum()) and nf > 150
    # the reference's bookkeeping: a MapPoint that lost its key point to a later one was Replace()d by it, so it still resolves to the same index
    assert np.array_equal(np.where(fused, bi, -1), idx)
    assert valid.mean() > 0.5 and len(set(level.tolist())) >= 5


@pytest.mark.parametrize("seed,ori", [(0, False), (1, True), (2, False)])
def test_search_for_triangulation(oracle, cam, gold, seed, ori):
    cp, r = cam
    s = synth.mapping_pair(10 + seed, n=1500, faceW=650)
    n2, m2, Ow1 = gold.value("triangulation_%d" % seed, lambda: r.search_for_triangulation(s["kCur"], s["dCur"], s["TcwCur"], s["hasMPCur"], s["nodeCur"], s["kLast"],
                                                                                           s["dLast"], s["TcwLast"], s["hasMPObs"], s["nodeObs"], s["E12"], ori))
    rays1, _ = oracle.key_point_rays(s["kCur"], 650, 650); rays2, _ = oracle.key_point_rays(s["kLast"], 650, 650)
    n1, m1 = oracle.search_for_triangulation(s["kCur"], s["dCur"], rays1, s["hasMPCur"], s["nodeCur"], s["kLast"], s["dLast"], rays2, s["hasMPObs"], s["nodeObs"], Ow1,
                                             s["TcwLast"], s["E12"], s["scale"], s["level_sigma2"], 650, 650, ori)
    assert n1 == n2 and n1 > 100
    assert np.array_equal(m1, m2)
    good = m1 >= 0
    assert (s["src"][good] == m1[good]).mean() > 0.9


def test_fuse_on_face_boundaries(oracle, cam, gold):
    """TransformRaysToCubemap leaves in-face coordinates (no tile offset) in (u, v) when its in-face bounds test fails, and Fuse does not look at the
    returned face - it only asks IsInImage(u, v) (src/ORBMatcher.cpp:1150-1154). MapPoints exactly on a face seam (|x/z| == 1 etc.) and behind the
    camera exercise that path: oracle == compiled reference."""
    cp, r = cam
    s = synth.mapping_pair(5, n=1200, faceW=650)
    rng = np.random.default_rng(11)
    Xw = s["Xw"].copy()
    n = len(Xw)
    d = rng.uniform(2.0, 9.0, n).astype(np.float32); y = rng.uniform(-0.9, 0.9, n).astype(np.float32) * d
    k = np.arange(n) % 6
    Xw[k == 0] = np.stack([d, y, d], 1)[k == 0]           # x / z == 1: front test passes, u == W fails the in-face test
    Xw[k == 1] = np.stack([-d, y, d], 1)[k == 1]          # x / z == -1
    Xw[k == 2] = np.stack([y, d, d], 1)[k == 2]           # y / z == 1
    Xw[k == 3] = np.stack([d, y, -d], 1)[k == 3]          # behind: right face, z / x == -1
    Xw[k == 4] = 0                                        # the origin: no face at all -> (-1, -1)
    I4 = np.eye(4, dtype=np.float32)
    nf, valid, level, idx = gold.value("fuse_boundaries", lambda: r.fuse(s["kCur"], s["dCur"], I4, Xw, s["kLast"], s["dLast"], I4, 4.0))
    g = oracle.FrameGrid(s["kCur"], 650, 650)
    bi, bd = g.fuse_search(s["dCur"], I4, s["scale"], s["inv_level_sigma2"], valid, Xw, level, s["dLast"], 4.0)
    fused = bd <= 50
    assert nf == int(fused.sum())
    assert np.array_equal(np.where(fused, bi, -1), idx)
