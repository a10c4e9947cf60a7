"""oracle (CPU restatement)  ==  oracle/_ref/libref.so (the reference's own sources compiled unmodified against the cv:: shim).

This is what pins the oracle to the reference: with the two environment pins on (monotonic node allocator, det_sincos; see
oracle/ref_api.cpp) the reference code is deterministic and must equal the restatement bit for bit. The unpinned runs QUANTIFY the
reference's own non-determinism (heap-address tie-break in DistributeOctTree, glibc sincosf, gcc FMA contraction).
The reference's results are read from tests/golden/ref_oracle_ref.npz (tests/refgold.py)."""
import os

import numpy as np
import pytest

from cubemapslam_b200 import config, synth
from oracle import ref
from tests.refgold import RECORD, gold  # noqa: F401

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _bits(a, b):
    return int(np.unpackbits(a ^ b).sum())


@pytest.fixture(scope="module")
def lafida(oracle):
    cfg = config.lafida_450()
    cp = oracle.cam_params(cfg)
    return cfg, cp, config.load_mask("gray_lafida_cubemap_mask_450"), oracle.build_maps(cp)


def test_camera_maps_and_warp(oracle, lafida, gold):
    cfg, cp, mask, (m1, m2) = lafida
    r = ref.Ref(cp) if RECORD else None
    # CamModelGeneral::CubemapToFisheye of the reference, per canvas pixel
    assert gold.same("maps", (m1, m2), lambda: r.build_maps())
    fr = synth.fisheye_frame(cfg, 2)
    assert gold.same("warp", oracle.warp(cp, fr, m1, m2), lambda: r.warp(fr, *r.build_maps()))
    rng = np.random.default_rng(3)
    probes = rng.uniform(-10, 1360, (50, 2))

    def ref_probes():
        out = np.zeros((len(probes), 2))
        for i, (up, vp) in enumerate(probes):
            uf = np.zeros(1); vf = np.zeros(1)
            r.L.ref_cubemap_to_fisheye(ref.C.c_double(up), ref.C.c_double(vp), ref._p(uf), ref._p(vf))
            out[i] = (uf[0], vf[0])
        return out
    rp = gold.value("cubemap_to_fisheye", ref_probes)
    for (up, vp), b in zip(probes, rp):
        assert oracle.cubemap_to_fisheye(cp, float(up), float(vp)) == (b[0], b[1])


@pytest.mark.parametrize("frame_idx", [0, 1, 5])
def test_extractor_config1_bit_exact(oracle, lafida, gold, frame_idx):
    cfg, cp, mask, (m1, m2) = lafida
    canvas = oracle.warp(cp, synth.fisheye_frame(cfg, frame_idx), m1, m2)
    ex = oracle.ORBextractor(2000, 1.2, 8, 20, 7, 450, 450)
    k1, d1 = ex(canvas, mask)
    rex = ref.Ref(cp).extractor(2000, 1.2, 8, 20, 7) if RECORD else None
    k2, d2 = rex(canvas, mask) if RECORD else (None, None)
    for l in range(8):
        assert gold.same("level%d_frame%d" % (l, frame_idx), ex.level_image(l), lambda: rex.level_image(l)), "pyramid level %d" % l
    assert len(k1) == gold.value("n_frame%d" % frame_idx, lambda: len(k2)) > 1000
    assert gold.same("kps_frame%d" % frame_idx, k1, lambda: k2), "keypoints (x, y, size, angle, response, octave, order)"
    assert gold.same("desc_frame%d" % frame_idx, d1, lambda: d2), "descriptors"


def test_extractor_config2_bit_exact_and_golden(oracle, gold):
    cfg = config.front_1024()
    mask = config.load_mask("gray_cubemap_front_mask_650")
    cp = oracle.cam_params(cfg)
    m1, m2 = oracle.build_maps(cp)
    canvas = oracle.warp(cp, synth.fisheye_frame(cfg, 7), m1, m2)
    k1, d1 = oracle.ORBextractor(3000, 1.2, 8, 20, 7, 650, 650)(canvas, mask)
    k2, d2 = ref.Ref(cp).extractor(3000, 1.2, 8, 20, 7)(canvas, mask) if RECORD else (None, None)
    assert len(k1) == gold.value("n_config2", lambda: len(k2)) > 1500 and gold.same("config2", (k1, d1), lambda: (k2, d2))
    g = np.load(os.path.join(GOLD, "ref_extract_front650_frame7.npz"))
    assert np.array_equal(g["kps"].view(np.uint8), k1.view(np.uint8)) and np.array_equal(g["desc"], d1)


def test_reference_golden_equals_oracle_golden():
    a = np.load(os.path.join(GOLD, "extract_lafida450_frame0.npz")); b = np.load(os.path.join(GOLD, "ref_extract_lafida450_frame0.npz"))
    assert np.array_equal(a["kps"].view(np.uint8), b["kps"].view(np.uint8)) and np.array_equal(a["desc"], b["desc"])


def test_degenerate_and_textured_corner(oracle, lafida, gold):
    cfg, cp, mask, (m1, m2) = lafida
    r = ref.Ref(cp) if RECORD else None
    flat = oracle.warp(cp, np.full((cp.Ih, cp.Iw), 200, np.uint8), m1, m2)
    rng = np.random.default_rng(0)
    tex = oracle.warp(cp, synth.fisheye_frame(cfg, 5), m1, m2); tex[:450, :450] = rng.integers(0, 256, (450, 450), dtype=np.uint8)
    for i, (canvas, nf) in enumerate(((flat, 2000), (tex, 2000), (tex, 6000))):     # 6000 = the 3x nFeatures initialisation extractor (src/Tracking.cpp:96)
        k1, d1 = oracle.ORBextractor(nf, 1.2, 8, 20, 7, 450, 450)(canvas, mask)
        assert gold.same("case%d" % i, (k1, d1), lambda: r.extractor(nf, 1.2, 8, 20, 7)(canvas, mask))


def _sym(k):
    return set(zip(k["x"].tolist(), k["y"].tolist(), k["octave"].tolist()))


def test_unpinned_reference_drift_is_quantified(oracle, lafida, gold, capsys):
    """What the oracle's two definitions replace, measured on config 1 (reported, with loose bounds). The unpinned reference results are
    stored as their difference from the pinned reference's, which the oracle must equal bit for bit (checked first)."""
    cfg, cp, mask, (m1, m2) = lafida
    tot_bits = tot_desc = moved = tot_kp = fma_bits = 0
    for fi in range(4):
        canvas = oracle.warp(cp, synth.fisheye_frame(cfg, fi), m1, m2)
        k1, d1 = oracle.ORBextractor(2000, 1.2, 8, 20, 7, 450, 450)(canvas, mask)
        assert gold.same("pinned_frame%d" % fi, (k1, d1), lambda: ref.Ref(cp).extractor(2000, 1.2, 8, 20, 7)(canvas, mask))

        def desc_diff(**kw):                # (changed byte index, xor) of the unpinned reference's descriptors; keypoints must be unchanged
            k, d = ref.Ref(cp, pins=ref.PIN_ALLOC, **kw).extractor(2000, 1.2, 8, 20, 7)(canvas, mask)
            assert np.array_equal(k1.view(np.uint8), k.view(np.uint8))
            x = (d1 ^ d).reshape(-1)
            return np.nonzero(x)[0].astype(np.int32), x[x != 0]
        # (a) glibc sincosf instead of det_sincos (allocator still pinned): same keypoints, count differing descriptor bits
        at, xor = gold.value("sincosf_frame%d" % fi, desc_diff)
        d2 = d1.copy().reshape(-1); d2[at] ^= xor
        tot_bits += _bits(d1.reshape(-1), d2); tot_desc += d1.size * 8
        # (b) gcc's default FMA contraction in the reference code (CMakeLists.txt: -O3 -march=native), glibc sincosf
        at, xor = gold.value("fma_frame%d" % fi, lambda: desc_diff(variant="libref_fma.so"))
        d3 = d1.copy().reshape(-1); d3[at] ^= xor
        fma_bits += _bits(d1.reshape(-1), d3)
        # (c) glibc malloc instead of the monotonic node arena: DistributeOctTree's sort by (count, heap address); stored as the keypoints
        # (x, y, octave) in the symmetric difference with the pinned run
        sd = gold.value("malloc_frame%d" % fi, lambda: np.array(sorted(_sym(k1) ^ _sym(ref.Ref(cp, pins=ref.PIN_SINCOS).extractor(2000, 1.2, 8, 20, 7)(canvas, mask)[0])),
                                                                  np.float64).reshape(-1, 3))
        s1 = _sym(k1); s4 = s1 ^ set((float(x), float(y), int(o)) for x, y, o in sd)
        moved += len(s1 ^ s4); tot_kp += len(k1)
    with capsys.disabled():
        print("\n[oracle vs stock reference build, 4 frames of config 1] glibc sincosf: %d of %d descriptor bits differ; +FMA contraction: %d bits; "
              "glibc malloc tie-break: %d keypoints of %d in the symmetric difference" % (tot_bits, tot_desc, fma_bits, moved, tot_kp))
    assert tot_bits <= tot_desc * 1e-4 and fma_bits <= tot_desc * 1e-3 and moved <= 0.05 * tot_kp


def test_descriptor_distance_kat(oracle, lafida, gold):
    cfg, cp, mask, maps = lafida
    r = ref.Ref(cp) if RECORD else None
    z = np.zeros(32, np.uint8); o = np.full(32, 255, np.uint8)
    rng = np.random.default_rng(1)
    pairs = [(z, o), (o, o)] + [(rng.integers(0, 256, 32, dtype=np.uint8), rng.integers(0, 256, 32, dtype=np.uint8)) for _ in range(200)]
    rd = gold.value("distance", lambda: np.array([r.descriptor_distance(a, b) for a, b in pairs], np.int32))
    assert rd[0] == 256 and rd[1] == 0
    for (a, b), d in zip(pairs[2:], rd[2:]):
        assert d == oracle.descriptor_distance(a, b) == int(np.unpackbits(a ^ b).sum())


def test_shim_gemm_matches_cv2(lafida, gold):
    """`R*x+t` and `-R.t()*t` as evaluated by the cv:: shim under the compiled reference == cv2.gemm 4.13 (small-matrix float path /
    transposed double path); every projection of the matcher path goes through these two expressions."""
    cv2 = pytest.importorskip("cv2")
    cfg, cp, mask, maps = lafida
    rng = np.random.default_rng(0)
    cases = []
    for _ in range(3000):
        R = rng.normal(0, 1, (3, 3)).astype(np.float32); x = rng.normal(0, 5, (3, 1)).astype(np.float32); t = rng.normal(0, 3, (3, 1)).astype(np.float32)
        cases.append((R, x, t))

    def shim():
        L = ref.Ref(cp).L
        out = np.zeros((len(cases), 2, 3), np.float32)
        for i, (R, x, t) in enumerate(cases):
            L.ref_expr_Rx_plus_t(ref._p(R), ref._p(x), ref._p(t), ref._p(out[i, 0]))
            L.ref_expr_neg_Rt_t(ref._p(R), ref._p(t), ref._p(out[i, 1]))
        return out
    want = np.stack([np.stack([cv2.gemm(R, x, 1.0, t, 1.0)[:, 0], cv2.gemm(R, t, -1.0, None, 0.0, flags=cv2.GEMM_1_T)[:, 0]]) for R, x, t in cases])
    assert gold.same("gemm", want.astype(np.float32), shim)
