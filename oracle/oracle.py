"""ctypes wrapper around oracle/liboracle.so (ORACLE: test infrastructure, not product code)."""
import ctypes as C
import os
import subprocess
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

KP_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"),
                     ("octave", "<i4"), ("class_id", "<i4")])


class CamParams(C.Structure):
    _fields_ = [("c", C.c_double), ("d", C.c_double), ("e", C.c_double), ("u0", C.c_double), ("v0", C.c_double),
                ("p", C.c_double * 5), ("invp", C.c_double * 12), ("Iw", C.c_int), ("Ih", C.c_int),
                ("faceW", C.c_int), ("faceH", C.c_int), ("fov", C.c_double)]


def cam_params(cfg):
    """cfg: dict with the reference YAML keys (Camera.*, CubeFace.*)."""
    cp = CamParams()
    cp.c, cp.d, cp.e = cfg["Camera.c"], cfg["Camera.d"], cfg["Camera.e"]
    cp.u0, cp.v0 = cfg["Camera.u0"], cfg["Camera.v0"]
    for i in range(5):
        cp.p[i] = cfg.get("Camera.a%d" % i, 0.0) if i < int(cfg["Camera.nrpol"]) else 0.0
    for i in range(12):
        cp.invp[i] = cfg.get("Camera.pol%d" % i, 0.0) if i < int(cfg["Camera.nrinvpol"]) else 0.0
    cp.Iw, cp.Ih = int(cfg["Camera.Iw"]), int(cfg["Camera.Ih"])
    cp.faceW, cp.faceH = int(cfg["CubeFace.w"]), int(cfg["CubeFace.h"])
    cp.fov = cfg["Camera.fov"]
    return cp


def build():
    subprocess.check_call(["make", "-s", "-C", _HERE, "liboracle.so"])
    # oracle/_ref (the reference's own sources against the cv:: shim) can only be built where the reference tree exists
    if os.path.isdir(os.environ.get("REF", "/root/reference")):
        subprocess.check_call(["make", "-s", "-j8", "-C", _HERE, "ref"])


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "liboracle.so")
        if not os.path.exists(path):
            build()
        _LIB = C.CDLL(path)
        _LIB.orc_orb_create.restype = C.c_void_p
        _LIB.orc_warp_extract_batch.restype = C.c_long
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _u8(a):
    return np.ascontiguousarray(a, dtype=np.uint8)


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


# ----------------------------------------------------------------------------- primitives
def remap_bilinear(src, mapx, mapy):
    src = _u8(src); mapx = _f32(mapx); mapy = _f32(mapy)
    dst = np.empty(mapx.shape, np.uint8)
    lib().orc_remap_bilinear(_p(src), src.shape[1], src.shape[0], _p(mapx), _p(mapy), _p(dst), mapx.shape[1], mapx.shape[0])
    return dst


def resize_linear(src, dw, dh):
    src = _u8(src); dst = np.empty((dh, dw), np.uint8)
    lib().orc_resize_linear(_p(src), src.shape[1], src.shape[0], _p(dst), dw, dh)
    return dst


def fast(img, thr):
    img = _u8(img); cap = img.size
    out = np.empty((cap, 3), np.int32)
    n = lib().orc_fast(_p(img), img.shape[1], img.shape[0], int(thr), _p(out), cap)
    return out[:n].copy()


def gaussian7(img):
    img = _u8(img); dst = np.empty_like(img)
    lib().orc_gaussian7(_p(img), img.shape[1], img.shape[0], _p(dst))
    return dst


def fast_atan2(y, x):
    y = _f32(y); x = _f32(x); out = np.empty_like(y)
    lib().orc_fast_atan2(_p(y), _p(x), _p(out), y.size)
    return out


def sincos(a):
    a = _f32(a); s = np.empty_like(a); c = np.empty_like(a)
    lib().orc_sincos(_p(a), _p(s), _p(c), a.size)
    return s, c


# ----------------------------------------------------------------------------- warp
def build_maps(cp):
    W3, H3 = 3 * cp.faceW, 3 * cp.faceH
    m1 = np.empty((H3, W3), np.float32); m2 = np.empty((H3, W3), np.float32)
    lib().orc_build_maps(C.byref(cp), _p(m1), _p(m2))
    return m1, m2


def cubemap_to_fisheye(cp, up, vp):
    uf = C.c_double(); vf = C.c_double()
    lib().orc_cubemap_to_fisheye(C.byref(cp), C.c_double(up), C.c_double(vp), C.byref(uf), C.byref(vf))
    return uf.value, vf.value


def warp(cp, fisheye, m1, m2, canvas=None):
    fisheye = _u8(fisheye)
    assert fisheye.shape == (cp.Ih, cp.Iw)
    if canvas is None:
        canvas = np.zeros((3 * cp.faceH, 3 * cp.faceW), np.uint8)
    lib().orc_warp(C.byref(cp), _p(fisheye), _p(m1), _p(m2), _p(canvas))
    return canvas


# ----------------------------------------------------------------------------- extractor
class ORBextractor:
    def __init__(self, nfeatures, scaleFactor, nlevels, iniThFAST, minThFAST, faceW, faceH):
        self.nlevels = nlevels
        self.nfeatures = nfeatures
        self._h = C.c_void_p(lib().orc_orb_create(int(nfeatures), C.c_float(scaleFactor), int(nlevels), int(iniThFAST),
                                                  int(minThFAST), int(faceW), int(faceH)))
        sc = [np.empty(nlevels, np.float32) for _ in range(4)]
        per = np.empty(nlevels, np.int32); um = np.empty(16, np.int32)
        lib().orc_orb_tables(self._h, _p(sc[0]), _p(sc[1]), _p(sc[2]), _p(sc[3]), _p(per), _p(um))
        self.scale, self.inv_scale, self.sigma2, self.inv_sigma2 = sc
        self.features_per_level, self.umax = per, um

    def __del__(self):
        try:
            lib().orc_orb_destroy(self._h)
        except Exception:
            pass

    def __call__(self, image, mask):
        image = _u8(image); mask = _u8(mask)
        assert image.shape == mask.shape
        n = lib().orc_orb_extract(self._h, _p(image), image.shape[1], image.shape[0], _p(mask))
        kps = np.empty(n, KP_DTYPE); desc = np.empty((n, 32), np.uint8)
        lib().orc_orb_result(self._h, _p(kps), _p(desc))
        return kps, desc

    def level_image(self, level, blurred=False):
        w = C.c_int(); h = C.c_int()
        lib().orc_orb_level_size(self._h, level, C.byref(w), C.byref(h))
        out = np.zeros((h.value, w.value), np.uint8)
        lib().orc_orb_level_image(self._h, level, int(blurred), _p(out))
        return out

    def stage(self, level, stage):
        """stage 0: FAST-grid candidates (minBorder-relative); 1: after distribution + orientation (level coords)."""
        n = lib().orc_orb_stage_count(self._h, level, stage)
        out = np.empty(n, KP_DTYPE)
        lib().orc_orb_stage_get(self._h, level, stage, _p(out))
        return out


def warp_extract_batch(cp, fisheyes, m1, m2, mask, nfeatures, scaleFactor, nlevels, iniTh, minTh, nthreads):
    fisheyes = _u8(fisheyes); mask = _u8(mask)
    return lib().orc_warp_extract_batch(C.byref(cp), _p(fisheyes), fisheyes.shape[0], _p(m1), _p(m2), _p(mask), int(nfeatures),
                                        C.c_float(scaleFactor), int(nlevels), int(iniTh), int(minTh), int(nthreads))


def warp_extract_batch_out(cp, fisheyes, m1, m2, mask, nfeatures, scaleFactor, nlevels, iniTh, minTh, nthreads, cap):
    fisheyes = _u8(fisheyes); mask = _u8(mask); F = fisheyes.shape[0]
    kps = np.zeros((F, cap), KP_DTYPE); desc = np.zeros((F, cap, 32), np.uint8); n = np.zeros(F, np.int32)
    lib().orc_warp_extract_batch_out.restype = C.c_long
    lib().orc_warp_extract_batch_out(C.byref(cp), _p(fisheyes), F, _p(m1), _p(m2), _p(mask), int(nfeatures), C.c_float(scaleFactor), int(nlevels), int(iniTh), int(minTh),
                                     int(nthreads), int(cap), _p(kps), _p(desc), _p(n))
    return kps, desc, n


def match_frames_batch(kps, desc, n, nnratio=0.6, thLow=50, checkOri=True, nthreads=1):
    kps = np.ascontiguousarray(kps); desc = _u8(desc); n = _i32(n)
    F, stride = kps.shape
    m = np.full((max(F - 1, 1), stride), -1, np.int32); nm = np.zeros(max(F - 1, 1), np.int32)
    lib().orc_match_frames_batch.restype = C.c_long
    lib().orc_match_frames_batch(_p(kps), _p(desc), _p(n), stride, F, C.c_float(nnratio), int(thLow), int(checkOri), _p(m), _p(nm), int(nthreads))
    return nm, m


# ----------------------------------------------------------------------------- matcher
def descriptor_distance(a, b):
    a = _u8(a); b = _u8(b)
    return lib().orc_descriptor_distance(_p(a), _p(b))


def search_by_bow(descKF, angKF, kfValid, nodeKF, descF, angF, nodeF, nnratio=0.7, checkOri=True):
    descKF = _u8(descKF); descF = _u8(descF); angKF = _f32(angKF); angF = _f32(angF)
    kfValid = _u8(kfValid); nodeKF = _i32(nodeKF); nodeF = _i32(nodeF)
    matchF = np.empty(descF.shape[0], np.int32)
    n = lib().orc_search_by_bow(_p(descKF), _p(angKF), _p(kfValid), _p(nodeKF), descKF.shape[0], _p(descF), _p(angF), _p(nodeF),
                                descF.shape[0], C.c_float(nnratio), int(checkOri), _p(matchF))
    return n, matchF


def search_by_bow_kf(desc1, ang1, valid1, node1, desc2, ang2, valid2, node2, nnratio=0.75, checkOri=True):
    desc1 = _u8(desc1); desc2 = _u8(desc2); ang1 = _f32(ang1); ang2 = _f32(ang2)
    valid1 = _u8(valid1); valid2 = _u8(valid2); node1 = _i32(node1); node2 = _i32(node2)
    m = np.empty(desc1.shape[0], np.int32)
    n = lib().orc_search_by_bow_kf(_p(desc1), _p(ang1), _p(valid1), _p(node1), desc1.shape[0], _p(desc2), _p(ang2), _p(valid2), _p(node2), desc2.shape[0],
                                   C.c_float(nnratio), int(checkOri), _p(m))
    return n, m


def match_bruteforce(descA, angA, descB, angB, nnratio=0.6, thLow=50, checkOri=True):
    descA = _u8(descA); descB = _u8(descB); angA = _f32(angA); angB = _f32(angB)
    nA = descA.shape[0]
    m = np.empty(nA, np.int32); d = np.empty(nA, np.int32); s = np.empty(nA, np.int32)
    n = lib().orc_match_bruteforce(_p(descA), _p(angA), nA, _p(descB), _p(angB), descB.shape[0], C.c_float(nnratio), int(thLow),
                                   int(checkOri), _p(m), _p(d), _p(s))
    return n, m, d, s


def match_bruteforce_batch(descA, angA, descB, angB, nnratio=0.6, thLow=50, checkOri=True, nthreads=1):
    descA = _u8(descA); descB = _u8(descB); angA = _f32(angA); angB = _f32(angB)
    P, nA = descA.shape[0], descA.shape[1]
    m = np.empty((P, nA), np.int32); nm = np.empty(P, np.int32)
    lib().orc_match_bruteforce_batch(_p(descA), _p(angA), nA, _p(descB), _p(angB), descB.shape[1], P, C.c_float(nnratio), int(thLow),
                                     int(checkOri), _p(m), _p(nm), int(nthreads))
    return nm, m


# ----------------------------------------------------------------------------- per-frame indexing
def key_point_rays(kps, faceW, faceH):
    kps = np.ascontiguousarray(kps); n = len(kps)
    rays = np.zeros((n, 3), np.float32); faces = np.zeros(n, np.int32)
    lib().orc_key_point_rays(_p(kps), n, int(faceW), int(faceH), _p(rays), _p(faces))
    return rays, faces


class FrameGrid:
    """Frame::AssignFeaturesToGrid + GetFeaturesInArea (reference src/Frame.cpp:158-176,251-716)."""
    NCELLS = 5 * 50 * 50

    def __init__(self, kps, faceW, faceH):
        self.kps = np.ascontiguousarray(kps); self.n = len(self.kps)
        lib().orc_grid_create.restype = C.c_void_p
        self._h = C.c_void_p(lib().orc_grid_create(_p(self.kps), self.n, int(faceW), int(faceH)))

    def __del__(self):
        try:
            lib().orc_grid_destroy(self._h)
        except Exception:
            pass

    def csr(self):
        start = np.zeros(self.NCELLS + 1, np.int32); idx = np.zeros(max(self.n, 1), np.int32)
        m = lib().orc_grid_csr(self._h, _p(start), _p(idx))
        return start, idx[:m]

    def features_in_area(self, x, y, r, min_level=-1, max_level=-1):
        buf = np.empty(8192, np.int32)
        n = lib().orc_features_in_area(self._h, C.c_float(x), C.c_float(y), C.c_float(r), int(min_level), int(max_level), _p(buf), 8192)
        return buf[:n].copy()


    def search_by_projection_last(self, dCur, TcwCur, scale_factors, kLast, hasMP, Xw, dMP, mpObs, curTaken, cosFovTh, th, checkOri=True):
        """ORBMatcher::SearchByProjection(CurrentFrame, LastFrame, th, mono) (reference src/ORBMatcher.cpp:130-251); self = CurrentFrame's grid."""
        dCur = _u8(dCur); TcwCur = _f32(TcwCur).reshape(16); sf = _f32(scale_factors); kLast = np.ascontiguousarray(kLast)
        hasMP = _u8(hasMP); Xw = _f32(Xw); dMP = _u8(dMP); mpObs = _i32(mpObs); curTaken = _u8(curTaken)
        match = np.empty(self.n, np.int32)
        n = lib().orc_search_by_projection_last(self._h, _p(dCur), _p(TcwCur), _p(sf), _p(kLast), len(kLast), _p(hasMP), _p(Xw), _p(dMP), _p(mpObs), _p(curTaken),
                                                C.c_float(cosFovTh), C.c_float(th), int(checkOri), _p(match))
        return n, match

    def search_by_projection_local(self, dF, scale_factors, inView, projXY, level, viewCos, dMP, mpObs, fTaken, th, nnratio):
        """ORBMatcher::SearchByProjection(F, vpMapPoints, th) (reference src/ORBMatcher.cpp:51-128); self = F's grid."""
        dF = _u8(dF); sf = _f32(scale_factors); inView = _u8(inView); projXY = _f32(projXY); level = _i32(level); viewCos = _f32(viewCos)
        dMP = _u8(dMP); mpObs = _i32(mpObs); fTaken = _u8(fTaken)
        match = np.empty(self.n, np.int32)
        n = lib().orc_search_by_projection_local(self._h, _p(dF), _p(sf), len(inView), _p(inView), _p(projXY), _p(level), _p(viewCos), _p(dMP), _p(mpObs), _p(fTaken),
                                                 C.c_float(th), C.c_float(nnratio), _p(match))
        return n, match


    def fuse_search(self, dKF, Tcw, scale_factors, inv_level_sigma2, valid, Xw, level, dMP, th):
        """The search of ORBMatcher::Fuse(pKF, vpMapPoints, th) (reference src/ORBMatcher.cpp:1126-1240); self = the KeyFrame's grid.
        Returns (bestIdx, bestDist) per MapPoint: the key point it would be fused with (-1 / 256: none)."""
        dKF = _u8(dKF); Tcw = _f32(Tcw).reshape(16); sf = _f32(scale_factors); isg = _f32(inv_level_sigma2); valid = _u8(valid); Xw = _f32(Xw); level = _i32(level); dMP = _u8(dMP)
        n = len(valid); bi = np.empty(n, np.int32); bd = np.empty(n, np.int32)
        lib().orc_fuse_search(self._h, _p(dKF), _p(Tcw), _p(sf), _p(isg), n, _p(valid), _p(Xw), _p(level), _p(dMP), C.c_float(th), _p(bi), _p(bd))
        return bi, bd


def distinctive_descriptors(desc, offset):
    """MapPoint::ComputeDistinctiveDescriptors (reference src/MapPoint.cpp:243-303) for a batch of MapPoints: desc = all observation descriptors,
    offset[p]..offset[p+1] = the rows of point p (in the order the reference iterates mObservations). Returns the chosen row per point (-1: none)."""
    desc = _u8(desc).reshape(-1, 32); offset = _i32(offset); n = len(offset) - 1
    best = np.empty(n, np.int32)
    lib().orc_distinctive_descriptors(_p(desc), _p(offset), n, _p(best))
    return best


def search_for_triangulation(k1, d1, rays1, hasMP1, node1, k2, d2, rays2, hasMP2, node2, Ow1, Tcw2, E12, scale_factors, level_sigma2, faceW, faceH, checkOri=True):
    """ORBMatcher::SearchForTriangulation (reference src/ORBMatcher.cpp:971-1124). Returns (nmatches, match12)."""
    k1 = np.ascontiguousarray(k1); k2 = np.ascontiguousarray(k2); d1 = _u8(d1); d2 = _u8(d2); rays1 = _f32(rays1); rays2 = _f32(rays2)
    hasMP1 = _u8(hasMP1); hasMP2 = _u8(hasMP2); node1 = _i32(node1); node2 = _i32(node2)
    Ow1 = _f32(Ow1); Tcw2 = _f32(Tcw2).reshape(16); E12 = _f32(E12).reshape(9); sf = _f32(scale_factors); ls2 = _f32(level_sigma2)
    m = np.empty(len(k1), np.int32)
    n = lib().orc_search_for_triangulation(_p(k1), _p(d1), _p(rays1), _p(hasMP1), _p(node1), len(k1), _p(k2), _p(d2), _p(rays2), _p(hasMP2), _p(node2), len(k2), _p(Ow1), _p(Tcw2),
                                           _p(E12), _p(sf), _p(ls2), int(faceW), int(faceH), int(checkOri), _p(m))
    return n, m


def vector_sigma(kx, ky, normal_rig, faceW, faceH):
    lib().orc_vector_sigma.restype = C.c_float
    nr = _f32(normal_rig)
    return float(lib().orc_vector_sigma(C.c_float(kx), C.c_float(ky), _p(nr), int(faceW), int(faceH)))


def area_rects(x, y, r, faceW, faceH):
    out = np.zeros((3, 5), np.int32)
    n = lib().orc_area_rects(C.c_float(x), C.c_float(y), C.c_float(r), int(faceW), int(faceH), _p(out))
    return out[:n].copy()


def ray_to_cubemap(xyz, faceW, faceH):
    xyz = _f32(xyz).reshape(-1, 3); n = len(xyz)
    uv = np.zeros((n, 2), np.float32); faces = np.zeros(n, np.int32)
    lib().orc_ray_to_cubemap(_p(xyz), n, int(faceW), int(faceH), _p(uv), _p(faces))
    return uv, faces


# ----------------------------------------------------------------------------- DBoW2 transform
class Vocabulary:
    """Vocabulary tree from flat arrays (nodes 1..n in file order: parent, leaf flag, descriptor, weight); transform like DBoW2 (levelsup 4)."""

    def __init__(self, k, L, parent, is_leaf, desc, weight):
        parent = _i32(parent); is_leaf = _u8(is_leaf); desc = _u8(desc); weight = np.ascontiguousarray(weight, np.float64)
        lib().orc_voc_create.restype = C.c_void_p
        self._h = C.c_void_p(lib().orc_voc_create(int(k), int(L), len(parent), _p(parent), _p(is_leaf), _p(desc), _p(weight)))

    def __del__(self):
        try:
            lib().orc_voc_destroy(self._h)
        except Exception:
            pass

    def transform(self, feats, levelsup=4):
        feats = _u8(feats); n = len(feats)
        bw = np.zeros(max(n, 1), np.int32); bv = np.zeros(max(n, 1), np.float64); node = np.zeros(max(n, 1), np.int32); word = np.zeros(max(n, 1), np.int32)
        m = lib().orc_voc_transform(self._h, _p(feats), n, int(levelsup), _p(bw), _p(bv), _p(node), _p(word))
        return bw[:m].copy(), bv[:m].copy(), node[:n].copy(), word[:n].copy()


# ----------------------------------------------------------------------------- bundle adjustment
def local_ba(Tcw, kf_fixed, pts, eMP, eKF, kpxy, inv_sigma2, faceW, faceH, its1=5, its2=10, stop_flag=None):
    Tcw = _f32(Tcw).copy(); pts = _f32(pts).copy()
    kf_fixed = _u8(kf_fixed); eMP = _i32(eMP); eKF = _i32(eKF); kpxy = _f32(kpxy); inv_sigma2 = _f32(inv_sigma2)
    nKF, nMP, nE = Tcw.shape[0], pts.shape[0], eMP.shape[0]
    outlier = np.zeros(nE, np.uint8); pose64 = np.zeros((nKF, 7)); pts64 = np.zeros((nMP, 3)); log = np.zeros((64, 4))
    sf = _p(stop_flag) if stop_flag is not None else None
    n = lib().orc_local_ba(nKF, nMP, nE, _p(Tcw), _p(kf_fixed), _p(pts), _p(eMP), _p(eKF), _p(kpxy), _p(inv_sigma2), int(faceW), int(faceH),
                           sf, int(its1), int(its2), _p(outlier), _p(pose64), _p(pts64), _p(log), 64)
    return dict(Tcw=Tcw.reshape(nKF, 4, 4), pts=pts, outlier=outlier, pose64=pose64, pts64=pts64, log=log[:n], iters=n)


def pose_opt(Tcw, Xw, kpxy, inv_sigma2, faceW, faceH):
    Tcw = _f32(Tcw).copy().reshape(16); Xw = _f32(Xw); kpxy = _f32(kpxy); inv_sigma2 = _f32(inv_sigma2)
    n = Xw.shape[0]
    outlier = np.zeros(max(n, 1), np.uint8); pose64 = np.zeros(7); log = np.zeros((64, 4)); nit = C.c_int()
    inl = lib().orc_pose_opt(n, _p(Tcw), _p(Xw), _p(kpxy), _p(inv_sigma2), int(faceW), int(faceH), _p(outlier), _p(pose64), _p(log), 64,
                             C.byref(nit))
    return dict(inliers=inl, Tcw=Tcw.reshape(4, 4), outlier=outlier[:n], pose64=pose64, log=log[:nit.value])


def ldlt_solve(S, g):
    """The dense LDL^T (no pivoting) local_ba solves its reduced camera system with; only the lower triangle of S is read.
    Returns (x, ok); ok is False on a zero / non-finite pivot."""
    S = np.ascontiguousarray(S, np.float64); g = np.ascontiguousarray(g, np.float64); n = len(g)
    assert S.shape == (n, n)
    x = np.zeros(n)
    ok = lib().orc_ldlt_solve(_p(S), n, _p(g), _p(x))
    return x, bool(ok)


def se3_exp(u):
    u = np.ascontiguousarray(u, np.float64); out = np.zeros(7)
    lib().orc_se3_exp(_p(u), _p(out))
    return out


def edge_eval(Tcw, X, kx, ky, faceW, faceH):
    Tcw = _f32(Tcw).reshape(16); X = np.ascontiguousarray(X, np.float64)
    err = np.zeros(2); Jp = np.zeros((2, 6)); Jx = np.zeros((2, 3)); face = C.c_int()
    lib().orc_edge_eval(_p(Tcw), _p(X), C.c_float(kx), C.c_float(ky), int(faceW), int(faceH), _p(err), _p(Jp), _p(Jx), C.byref(face))
    return err, Jp, Jx, face.value
