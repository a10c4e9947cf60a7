"""Host-side mirror of the reference Optimizer interface (reference include/Optimizer.h:42-63) on top of the C ABI.

  Optimizer.LocalBundleAdjustment   src/Optimizer.cpp:192-451 (the local window is passed as flat arrays)
  Optimizer.PoseOptimization        src/Optimizer.cpp:48-190  (batched over independent frames)
Multi-GPU: init_nccl(rank, nranks, id) shards the landmarks (l % nranks) and all-reduces the reduced camera system."""
import ctypes as C

import numpy as np

from ._capi import BAProblem, BAResult, check, lib, ptr


class Optimizer:
    def __init__(self, device=0):
        self._h = C.c_void_p()
        check(lib().cslam_optimizer_create(C.byref(self._h), int(device)))

    def close(self):
        if getattr(self, "_h", None):
            lib().cslam_optimizer_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launches(self):
        return lib().cslam_optimizer_launches(self._h)

    def set_timing(self, on):
        check(lib().cslam_optimizer_set_timing(self._h, int(bool(on))))

    def timing(self):
        out = {}
        for k in range(10):
            name = C.c_char_p(); ms = C.c_double(); cnt = C.c_int64()
            check(lib().cslam_optimizer_get_timing(self._h, k, C.byref(name), C.byref(ms), C.byref(cnt)))
            if cnt.value:
                out[name.value.decode()] = (ms.value, cnt.value)
        return out

    def solve_dense(self, Sg, stage=-1, cluster=0):
        """The reduced-camera-system solve of LocalBundleAdjustment on its own (test / measurement hook): Sg is (n+1) x n float64, S with the
        right-hand side as row n; only the lower triangle of S is read. Returns (x, failed)."""
        Sg = np.ascontiguousarray(Sg, np.float64)
        n = Sg.shape[1]
        if Sg.shape != (n + 1, n):
            raise ValueError("Sg must be (n+1) x n, got %s" % (Sg.shape,))
        x = np.empty(n); failed = C.c_int32()
        check(lib().cslam_ba_solve_dense(self._h, int(n), ptr(Sg), int(stage), int(cluster), ptr(x), C.byref(failed)))
        return x, bool(failed.value)

    @staticmethod
    def nccl_unique_id():
        buf = np.zeros(128, np.uint8)
        check(lib().cslam_nccl_unique_id(ptr(buf)))
        return buf

    def init_nccl(self, id128, rank, nranks):
        id128 = np.ascontiguousarray(id128, np.uint8)
        check(lib().cslam_optimizer_init_nccl(self._h, ptr(id128), int(rank), int(nranks)))

    def LocalBundleAdjustment(self, Tcw, kf_fixed, pts, eMP, eKF, kpxy, inv_sigma2, faceW, faceH, its1=5, its2=10, stop_flag=None):
        Tcw = np.ascontiguousarray(Tcw, np.float32).reshape(-1, 16).copy(); pts = np.ascontiguousarray(pts, np.float32).copy()
        kf_fixed = np.ascontiguousarray(kf_fixed, np.uint8); eMP = np.ascontiguousarray(eMP, np.int32); eKF = np.ascontiguousarray(eKF, np.int32)
        kpxy = np.ascontiguousarray(kpxy, np.float32); inv_sigma2 = np.ascontiguousarray(inv_sigma2, np.float32)
        nKF, nMP, nE = Tcw.shape[0], pts.shape[0], eMP.shape[0]
        p = BAProblem(nKF, nMP, nE, ptr(Tcw).value, ptr(kf_fixed).value, ptr(pts).value, ptr(eMP).value, ptr(eKF).value, ptr(kpxy).value,
                      ptr(inv_sigma2).value, int(faceW), int(faceH))
        outlier = np.zeros(max(nE, 1), np.uint8); pose64 = np.zeros((nKF, 7)); pts64 = np.zeros((max(nMP, 1), 3)); log = np.zeros((64, 4))
        r = BAResult(ptr(outlier).value, ptr(pose64).value, ptr(pts64).value, ptr(log).value, 64, 0, 0)
        sf = ptr(stop_flag) if stop_flag is not None else None
        check(lib().cslam_local_ba(self._h, C.byref(p), sf, int(its1), int(its2), C.byref(r)))
        return dict(Tcw=Tcw.reshape(nKF, 4, 4), pts=pts, outlier=outlier[:nE], pose64=pose64, pts64=pts64[:nMP], log=log[:r.iterations], iters=r.iterations,
                    trials=r.trials)

    @property
    def stream(self):
        lib().cslam_optimizer_stream.restype = C.c_void_p
        return lib().cslam_optimizer_stream(self._h)

    def sync(self):
        check(lib().cslam_optimizer_sync(self._h))

    def pose_optimization_dev(self, nframes, stride, count, Tcw, Xw, kpxy, inv_sigma2, faceW, faceH, outlier, inliers):
        check(lib().cslam_pose_optimization_dev(self._h, int(nframes), int(stride), ptr(count), ptr(Tcw), ptr(Xw), ptr(kpxy), ptr(inv_sigma2), int(faceW), int(faceH), ptr(outlier),
                                                ptr(inliers)))

    def PoseOptimization(self, Tcw, Xw, kpxy, inv_sigma2, faceW, faceH, offset=None):
        """Single frame (Tcw 4x4, Xw n x 3, ...) or a batch (Tcw F x 4 x 4, offset F+1 into the concatenated correspondences)."""
        Tcw = np.ascontiguousarray(Tcw, np.float32)
        single = Tcw.ndim == 2
        T = Tcw.reshape(-1, 16).copy()
        Xw = np.ascontiguousarray(Xw, np.float32).reshape(-1, 3); kpxy = np.ascontiguousarray(kpxy, np.float32).reshape(-1, 2)
        inv_sigma2 = np.ascontiguousarray(inv_sigma2, np.float32)
        if offset is None:
            offset = np.array([0, Xw.shape[0]], np.int32)
        offset = np.ascontiguousarray(offset, np.int32)
        F = T.shape[0]; n = int(offset[-1])
        outlier = np.zeros(max(n, 1), np.uint8); inl = np.zeros(F, np.int32); pose64 = np.zeros((F, 7))
        check(lib().cslam_pose_optimization(self._h, F, ptr(offset), ptr(T), ptr(Xw), ptr(kpxy), ptr(inv_sigma2), int(faceW), int(faceH), ptr(outlier), ptr(inl),
                                            ptr(pose64)))
        if single:
            return dict(inliers=int(inl[0]), Tcw=T.reshape(4, 4), outlier=outlier[:n], pose64=pose64[0])
        return dict(inliers=inl, Tcw=T.reshape(F, 4, 4), outlier=outlier[:n], pose64=pose64)
