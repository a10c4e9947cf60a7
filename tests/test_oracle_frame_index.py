"""oracle/frame_index.h (rays, 5x50x50 grid, GetFeaturesInArea with its cube-face wrap-around cases) == the reference's own Frame code
compiled in oracle/_ref/libref.so (src/Frame.cpp:158-176,251-716,728-760, include/CamModelGeneral.h:494-513).
The reference's results are read from tests/golden/ref_oracle_frame_index.npz (tests/refgold.py)."""
import numpy as np
import pytest

from cubemapslam_b200 import config, synth
from oracle import ref
from tests.refgold import RECORD, gold  # noqa: F401


@pytest.fixture(scope="module", params=[("lafida", 450), ("front", 650)])
def frame(request, oracle, gold):
    """(name, face width, key points, the reference's Frame or None): the key points are the oracle's, bit-identical to the reference Frame's."""
    name, W = request.param
    if name == "lafida":
        cfg = config.lafida_450(); mask = config.load_mask("gray_lafida_cubemap_mask_450"); nf = 2000
    else:
        cfg = config.front_1024(); mask = np.full((1950, 1950), 255, np.uint8); nf = 3000      # full mask: features near every face seam
    cp = oracle.cam_params(cfg)
    m1, m2 = oracle.build_maps(cp)
    kps, _ = oracle.ORBextractor(nf, 1.2, 8, 20, 7, W, W)(oracle.warp(cp, synth.fisheye_frame(cfg, 2), m1, m2), mask)
    F = None
    if RECORD:
        r = ref.Ref(cp)
        m1, m2 = r.build_maps()
        F = ref.RefFrame(r.extractor(nf, 1.2, 8, 20, 7), r.warp(synth.fisheye_frame(cfg, 2), m1, m2), mask)
    assert gold.same("kps_" + name, kps, lambda: F.kps)
    return name, W, kps, F


def test_rays_and_grid(oracle, frame, gold):
    name, W, kps, F = frame
    rays, faces = oracle.key_point_rays(kps, W, W)
    assert gold.same("rays_" + name, rays, lambda: F.rays)    # bit-exact unit bearing vectors
    g = oracle.FrameGrid(kps, W, W)
    start, idx = g.csr()
    assert len(idx) == gold.value("n_" + name, lambda: F.N) == gold.value("grid_count_" + name, lambda: F.grid_count).sum()
    assert np.array_equal(np.diff(start).reshape(5, 50, 50), gold.value("grid_count_" + name, lambda: F.grid_count))
    rng = np.random.default_rng(0)
    cells = [(rng.integers(0, 5), rng.integers(0, 50), rng.integers(0, 50)) for _ in range(300)]

    def lengths_then_indices(rows):                           # every queried cell: its length, then its key point indices
        return np.concatenate([np.concatenate([[len(b)], b]) for b in rows]).astype(np.int32)
    mine = lengths_then_indices(idx[start[k]:start[k + 1]] for k in ((f * 50 + c) * 50 + r_ for f, c, r_ in cells))
    assert gold.same("grid_cells_" + name, mine, lambda: lengths_then_indices(F.grid_cell(f, c, r_) for f, c, r_ in cells))


def test_features_in_area_all_wraparound_cases(oracle, frame, gold):
    name, W, kps, F = frame
    g = oracle.FrameGrid(kps, W, W)
    rng = np.random.default_rng(1)
    tiles = {0: (1, 1), 1: (0, 1), 2: (2, 1), 3: (1, 0), 4: (1, 2)}
    queries = []
    for face, (tc, tr) in tiles.items():
        for k in range(1500):
            # uniform in the face, with half of the samples pushed against an edge / a corner so that every overflow case is exercised
            u, v = rng.uniform(0, W, 2)
            mode = k % 4
            if mode >= 1:
                u = rng.choice([rng.uniform(0, 40), rng.uniform(W - 40, W - 0.01)])
            if mode >= 2:
                v = rng.choice([rng.uniform(0, 40), rng.uniform(W - 40, W - 0.01)])
            if mode == 3:
                u, v = v, u
            x = np.float32(tc * W + u); y = np.float32(tr * W + v)
            r = np.float32(rng.choice([7.0, 15.0, 15.0 * 1.728, 40.0, 75.0]))
            lv = int(rng.integers(0, 8)); lo, hi = [(-1, -1), (lv - 1, lv), (lv - 1, lv + 1), (0, 3)][k % 4]
            queries.append((x, y, r, lo, hi))
    queries.append((np.float32(10.0), np.float32(10.0), np.float32(30.0), -1, -1))     # a centre outside the five faces returns nothing

    def lengths_and_indices(fn):
        res = [np.asarray(fn(*q), np.int32) for q in queries]
        return np.array([len(a) for a in res], np.int32), np.concatenate(res)
    mine = lengths_and_indices(g.features_in_area)
    assert gold.same("features_in_area_" + name, mine, lambda: lengths_and_indices(F.features_in_area))
    assert mine[0][-1] == 0
    assert (mine[0][:-1] > 0).sum() > 0.2 * (len(queries) - 1)
