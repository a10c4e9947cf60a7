// ORACLE (test infrastructure, not product code): flat C entry points for oracle/oracle.py (ctypes).
// Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load this.
#include <cstring>
#include <memory>
#include <thread>
#include "ba.h"
#include "cam_model.h"
#include "bow.h"
#include "cvprim.h"
#include "frame_index.h"
#include "mapping.h"
#include "orb_extractor.h"
#include "orb_matcher.h"

using namespace orc;

extern "C" {

// ---- primitives (pinned against cv2 4.13 in tests/test_oracle_cv2.py)
void orc_remap_bilinear(const uint8_t* src, int sw, int sh, const float* mx, const float* my, uint8_t* dst, int dw, int dh) {
    remap_bilinear(src, sw, sh, sw, mx, my, dw, dst, dw, dh, dw);
}
void orc_resize_linear(const uint8_t* src, int sw, int sh, uint8_t* dst, int dw, int dh) { resize_linear(src, sw, sh, sw, dst, dw, dh, dw); }
int orc_fast(const uint8_t* img, int w, int h, int thr, int* xyr, int cap) {
    std::vector<FastKp> k; fast_nms(img, w, h, w, thr, k);
    int n = (int)k.size();
    for (int i = 0; i < n && i < cap; i++) { xyr[3 * i] = k[i].x; xyr[3 * i + 1] = k[i].y; xyr[3 * i + 2] = k[i].response; }
    return n;
}
void orc_gaussian7(const uint8_t* src, int w, int h, uint8_t* dst) { gaussian7(src, w, h, w, dst, w); }
void orc_fast_atan2(const float* y, const float* x, float* out, int n) { for (int i = 0; i < n; i++) out[i] = fast_atan2(y[i], x[i]); }
void orc_sincos(const float* a, float* s, float* c, int n) { for (int i = 0; i < n; i++) det_sincosf(a[i], &s[i], &c[i]); }

// ---- warp
void orc_build_maps(const CamParams* cp, float* map1, float* map2) { build_maps(*cp, map1, map2); }
void orc_cubemap_to_fisheye(const CamParams* cp, double up, double vp, double* uf, double* vf) { cubemap_to_fisheye(*cp, up, vp, *uf, *vf); }
void orc_warp(const CamParams* cp, const uint8_t* fisheye, const float* map1, const float* map2, uint8_t* canvas) {
    warp_fisheye_to_cubemap(*cp, fisheye, cp->Iw, map1, map2, canvas, 3 * cp->faceW);
}

// ---- extractor
struct OrbHandle { std::unique_ptr<ORBextractor> ex; std::vector<KeyPoint> kps; std::vector<uint8_t> desc; };
void* orc_orb_create(int nfeatures, float scaleFactor, int nlevels, int iniTh, int minTh, int faceW, int faceH) {
    OrbHandle* h = new OrbHandle; h->ex.reset(new ORBextractor(nfeatures, scaleFactor, nlevels, iniTh, minTh, faceW, faceH)); return h;
}
void orc_orb_destroy(void* h) { delete (OrbHandle*)h; }
void orc_orb_tables(void* hv, float* scale, float* invScale, float* sigma2, float* invSigma2, int* perLevel, int* umax) {
    ORBextractor& e = *((OrbHandle*)hv)->ex;
    for (int i = 0; i < e.nlevels; i++) { scale[i] = e.mvScaleFactor[i]; invScale[i] = e.mvInvScaleFactor[i]; sigma2[i] = e.mvLevelSigma2[i];
        invSigma2[i] = e.mvInvLevelSigma2[i]; perLevel[i] = e.mnFeaturesPerLevel[i]; }
    for (int i = 0; i < 16; i++) umax[i] = e.umax[i];
}
int orc_orb_extract(void* hv, const uint8_t* img, int cols, int rows, const uint8_t* mask) {
    OrbHandle* h = (OrbHandle*)hv; (*h->ex)(img, cols, rows, cols, mask, cols, h->kps, h->desc); return (int)h->kps.size();
}
void orc_orb_result(void* hv, KeyPoint* kps, uint8_t* desc) {
    OrbHandle* h = (OrbHandle*)hv;
    if (!h->kps.empty()) { std::memcpy(kps, h->kps.data(), h->kps.size() * sizeof(KeyPoint)); std::memcpy(desc, h->desc.data(), h->desc.size()); }
}
void orc_orb_level_size(void* hv, int level, int* w, int* hh) { const Image& L = ((OrbHandle*)hv)->ex->mvImagePyramid[level]; *w = L.w; *hh = L.h; }
void orc_orb_level_image(void* hv, int level, int blurred, uint8_t* out) {
    ORBextractor& e = *((OrbHandle*)hv)->ex; const Image& L = blurred ? e.mvBlurred[level] : e.mvImagePyramid[level];
    if (!L.px.empty()) std::memcpy(out, L.px.data(), L.px.size());
}
int orc_orb_stage_count(void* hv, int level, int stage) {
    ORBextractor& e = *((OrbHandle*)hv)->ex; return (int)(stage == 0 ? e.mvCandidates[level].size() : e.mvDistributed[level].size());
}
void orc_orb_stage_get(void* hv, int level, int stage, KeyPoint* out) {
    ORBextractor& e = *((OrbHandle*)hv)->ex; const std::vector<KeyPoint>& v = stage == 0 ? e.mvCandidates[level] : e.mvDistributed[level];
    if (!v.empty()) std::memcpy(out, v.data(), v.size() * sizeof(KeyPoint));
}
// timed CPU baseline: warp + extract over `nframes` fisheye frames with `nthreads` independent workers
// (each worker owns its extractor, like one reference process per core). Returns total keypoints.
long orc_warp_extract_batch(const CamParams* cp, const uint8_t* fisheyes, int nframes, const float* map1, const float* map2, const uint8_t* mask,
                            int nfeatures, float scaleFactor, int nlevels, int iniTh, int minTh, int nthreads) {
    std::vector<long> totals(nthreads, 0);
    auto work = [&](int t) {
        ORBextractor ex(nfeatures, scaleFactor, nlevels, iniTh, minTh, cp->faceW, cp->faceH);
        const int W3 = 3 * cp->faceW, H3 = 3 * cp->faceH;
        std::vector<uint8_t> canvas((size_t)W3 * H3, 0), desc; std::vector<KeyPoint> kps;
        for (int f = t; f < nframes; f += nthreads) {
            warp_fisheye_to_cubemap(*cp, fisheyes + (size_t)f * cp->Iw * cp->Ih, cp->Iw, map1, map2, canvas.data(), W3);
            ex(canvas.data(), W3, H3, W3, mask, W3, kps, desc);
            totals[t] += (long)kps.size();
        }
    };
    std::vector<std::thread> th;
    for (int t = 1; t < nthreads; t++) th.emplace_back(work, t);
    work(0);
    for (auto& x : th) x.join();
    long s = 0; for (long v : totals) s += v; return s;
}

// ---- matcher
int orc_descriptor_distance(const uint8_t* a, const uint8_t* b) { return descriptor_distance(a, b); }
int orc_search_by_bow(const uint8_t* descKF, const float* angKF, const uint8_t* kfValid, const int* nodeKF, int nKF, const uint8_t* descF,
                      const float* angF, const int* nodeF, int nF, float nnratio, int checkOri, int* matchF) {
    return search_by_bow(descKF, angKF, kfValid, nodeKF, nKF, descF, angF, nodeF, nF, nnratio, checkOri != 0, matchF);
}
int orc_search_by_bow_kf(const uint8_t* d1, const float* a1, const uint8_t* v1, const int* nd1, int n1, const uint8_t* d2, const float* a2, const uint8_t* v2,
                         const int* nd2, int n2, float nnratio, int checkOri, int* match12) {
    return search_by_bow_kf(d1, a1, v1, nd1, n1, d2, a2, v2, nd2, n2, nnratio, checkOri != 0, match12);
}
int orc_match_bruteforce(const uint8_t* descA, const float* angA, int nA, const uint8_t* descB, const float* angB, int nB, float nnratio,
                         int thLow, int checkOri, int* match12, int* dist12, int* second12) {
    return match_bruteforce(descA, angA, nA, descB, angB, nB, nnratio, thLow, checkOri != 0, match12, dist12, second12);
}
void orc_match_bruteforce_batch(const uint8_t* descA, const float* angA, int nA, const uint8_t* descB, const float* angB, int nB, int npairs,
                                float nnratio, int thLow, int checkOri, int* match12, int* nmatches, int nthreads) {
    auto work = [&](int t) {
        std::vector<int> d(nA), s(nA);
        for (int p = t; p < npairs; p += nthreads)
            nmatches[p] = match_bruteforce(descA + (size_t)p * nA * 32, angA + (size_t)p * nA, nA, descB + (size_t)p * nB * 32, angB + (size_t)p * nB, nB,
                                           nnratio, thLow, checkOri != 0, match12 + (size_t)p * nA, d.data(), s.data());
    };
    std::vector<std::thread> th;
    for (int t = 1; t < nthreads; t++) th.emplace_back(work, t);
    work(0);
    for (auto& x : th) x.join();
}

// all-pairs matching of consecutive frames (frame f vs f+1) in the front end's output layout, `nthreads` workers; returns total matches
long orc_match_frames_batch(const KeyPoint* kps, const uint8_t* desc, const int* n, int stride, int nframes, float nnratio, int thLow, int checkOri, int* match12, int* nmatches,
                            int nthreads) {
    std::vector<long> totals(nthreads, 0);
    auto work = [&](int t) {
        std::vector<float> aA(stride), aB(stride); std::vector<int> d(stride), s2(stride);
        for (int f = t; f + 1 < nframes; f += nthreads) {
            const int nA = n[f], nB = n[f + 1];
            for (int i = 0; i < nA; i++) aA[i] = kps[(size_t)f * stride + i].angle;
            for (int i = 0; i < nB; i++) aB[i] = kps[(size_t)(f + 1) * stride + i].angle;
            nmatches[f] = match_bruteforce(desc + (size_t)f * stride * 32, aA.data(), nA, desc + (size_t)(f + 1) * stride * 32, aB.data(), nB, nnratio, thLow, checkOri != 0,
                                           match12 + (size_t)f * stride, d.data(), s2.data());
            totals[t] += nmatches[f];
        }
    };
    std::vector<std::thread> th;
    for (int t = 1; t < nthreads; t++) th.emplace_back(work, t);
    work(0);
    for (auto& x : th) x.join();
    long s = 0; for (long v : totals) s += v; return s;
}
// warp + extract with per-frame outputs (for the extract+match CPU baseline): kps / desc: nframes x cap
long orc_warp_extract_batch_out(const CamParams* cp, const uint8_t* fisheyes, int nframes, const float* map1, const float* map2, const uint8_t* mask, int nfeatures, float scaleFactor,
                                int nlevels, int iniTh, int minTh, int nthreads, int cap, KeyPoint* kpsOut, uint8_t* descOut, int* nOut) {
    std::vector<long> totals(nthreads, 0);
    auto work = [&](int t) {
        ORBextractor ex(nfeatures, scaleFactor, nlevels, iniTh, minTh, cp->faceW, cp->faceH);
        const int W3 = 3 * cp->faceW, H3 = 3 * cp->faceH;
        std::vector<uint8_t> canvas((size_t)W3 * H3, 0), desc; std::vector<KeyPoint> kps;
        for (int f = t; f < nframes; f += nthreads) {
            warp_fisheye_to_cubemap(*cp, fisheyes + (size_t)f * cp->Iw * cp->Ih, cp->Iw, map1, map2, canvas.data(), W3);
            ex(canvas.data(), W3, H3, W3, mask, W3, kps, desc);
            const int m = std::min((int)kps.size(), cap);
            nOut[f] = m;
            if (m) { std::memcpy(kpsOut + (size_t)f * cap, kps.data(), (size_t)m * sizeof(KeyPoint)); std::memcpy(descOut + (size_t)f * cap * 32, desc.data(), (size_t)m * 32); }
            totals[t] += m;
        }
    };
    std::vector<std::thread> th;
    for (int t = 1; t < nthreads; t++) th.emplace_back(work, t);
    work(0);
    for (auto& x : th) x.join();
    long s = 0; for (long v : totals) s += v; return s;
}

// ---- per-frame indexing (rays, 5x50x50 grid) and windowed lookup
void orc_key_point_rays(const KeyPoint* kps, int n, int faceW, int faceH, float* rays, int* faces) {
    for (int i = 0; i < n; i++) { const int f = fi_pixel_to_ray(kps[i].x, kps[i].y, faceW, faceH, rays + 3 * i); if (faces) faces[i] = f; }
}
struct GridHandle { FrameGrid g; std::vector<KeyPoint> kps; };
void* orc_grid_create(const KeyPoint* kps, int n, int faceW, int faceH) {
    GridHandle* h = new GridHandle; h->kps.assign(kps, kps + n); h->g.build(h->kps.data(), n, faceW, faceH); return h;
}
void orc_grid_destroy(void* h) { delete (GridHandle*)h; }
// CSR view: cellStart[5*50*50+1], cellIdx[n] (cells in (face, col, row) order, indices ascending inside a cell)
int orc_grid_csr(void* hv, int* cellStart, int* cellIdx) {
    GridHandle* h = (GridHandle*)hv; int pos = 0;
    for (size_t c = 0; c < h->g.cells.size(); c++) { cellStart[c] = pos; for (int i : h->g.cells[c]) cellIdx[pos++] = i; }
    cellStart[h->g.cells.size()] = pos;
    return pos;
}
int orc_features_in_area(void* hv, float x, float y, float r, int minLevel, int maxLevel, int* out, int cap) {
    GridHandle* h = (GridHandle*)hv; std::vector<int> v;
    fi_features_in_area(h->g, h->kps.data(), x, y, r, minLevel, maxLevel, v);
    for (size_t i = 0; i < v.size() && (int)i < cap; i++) out[i] = v[i];
    return (int)v.size();
}

int orc_search_by_projection_last(void* hv, const uint8_t* dCur, const float* TcwCur, const float* scaleFactors, const KeyPoint* kLast, int nLast, const uint8_t* hasMP,
                                  const float* Xw, const uint8_t* dMP, const int* mpObs, const uint8_t* curTaken, float cosFovTh, float th, int checkOri, int* matchCur) {
    GridHandle* h = (GridHandle*)hv;
    return fi_search_by_projection_last(h->g, h->kps.data(), dCur, (int)h->kps.size(), TcwCur, scaleFactors, kLast, nLast, hasMP, Xw, dMP, mpObs, curTaken, cosFovTh, th,
                                        checkOri != 0, matchCur);
}
int orc_search_by_projection_local(void* hv, const uint8_t* dF, const float* scaleFactors, int nMP, const uint8_t* inView, const float* projXY, const int* level,
                                   const float* viewCos, const uint8_t* dMP, const int* mpObs, const uint8_t* fTaken, float th, float nnratio, int* matchF) {
    GridHandle* h = (GridHandle*)hv;
    return fi_search_by_projection_local(h->g, h->kps.data(), dF, (int)h->kps.size(), scaleFactors, nMP, inView, projXY, level, viewCos, dMP, mpObs, fTaken, th, nnratio, matchF);
}
// ---- LocalMapping feature operations (mapping.h)
void orc_distinctive_descriptors(const uint8_t* desc, const int* offset, int nPoints, int* best) {
    for (int p = 0; p < nPoints; p++) best[p] = distinctive_descriptor(desc + 32 * (size_t)offset[p], offset[p + 1] - offset[p]);
}
void orc_fuse_search(void* hv, const uint8_t* dKF, const float* Tcw, const float* scaleFactors, const float* invLevelSigma2, int nMP, const uint8_t* valid, const float* Xw,
                     const int* level, const uint8_t* dMP, float th, int* bestIdx, int* bestDist) {
    GridHandle* h = (GridHandle*)hv;
    fuse_search(h->g, h->kps.data(), dKF, Tcw, scaleFactors, invLevelSigma2, nMP, valid, Xw, level, dMP, th, bestIdx, bestDist);
}
int orc_search_for_triangulation(const KeyPoint* k1, const uint8_t* d1, const float* rays1, const uint8_t* hasMP1, const int* node1, int n1, const KeyPoint* k2, const uint8_t* d2,
                                 const float* rays2, const uint8_t* hasMP2, const int* node2, int n2, const float* Ow1, const float* Tcw2, const float* E12,
                                 const float* scaleFactors, const float* levelSigma2, int faceW, int faceH, int checkOri, int* match12) {
    return search_for_triangulation(k1, d1, rays1, hasMP1, node1, n1, k2, d2, rays2, hasMP2, node2, n2, Ow1, Tcw2, E12, scaleFactors, levelSigma2, faceW, faceH, checkOri != 0, match12);
}
float orc_vector_sigma(float kx, float ky, const float* normalRig, int faceW, int faceH) { return vector_sigma(kx, ky, normalRig, faceW, faceH); }

int orc_area_rects(float x, float y, float r, int faceW, int faceH, int* rects) {
    FiRect rc[3]; const float inv = static_cast<float>(3 * FI_G) / static_cast<float>((float)(3 * faceW) - 0.0f);
    const int n = fi_area_rects(x, y, r, faceW, faceH, inv, rc);
    for (int k = 0; k < n; k++) { rects[5 * k] = rc[k].face; rects[5 * k + 1] = rc[k].x0; rects[5 * k + 2] = rc[k].x1; rects[5 * k + 3] = rc[k].y0; rects[5 * k + 4] = rc[k].y1; }
    return n;
}
void orc_ray_to_cubemap(const float* xyz, int n, int faceW, int faceH, float* uv, int* faces) {
    for (int i = 0; i < n; i++) faces[i] = fi_ray_to_cubemap(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], faceW, faceH, uv[2 * i], uv[2 * i + 1]);
}

// ---- DBoW2 transform
void* orc_voc_create(int k, int L, int n, const int* parent, const uint8_t* isLeaf, const uint8_t* desc, const double* weight) {
    Vocabulary* v = new Vocabulary; v->build(k, L, n, parent, isLeaf, desc, weight); return v;
}
void orc_voc_destroy(void* v) { delete (Vocabulary*)v; }
int orc_voc_transform(void* vv, const uint8_t* feats, int n, int levelsup, int* bowWord, double* bowVal, int* nodeOf, int* wordOf) {
    std::vector<int> bw, no, wo; std::vector<double> bv;
    ((Vocabulary*)vv)->transform(feats, n, levelsup, bw, bv, no, wo);
    for (size_t i = 0; i < bw.size(); i++) { bowWord[i] = bw[i]; bowVal[i] = bv[i]; }
    for (int i = 0; i < n; i++) { nodeOf[i] = no[i]; wordOf[i] = wo[i]; }
    return (int)bw.size();
}

// ---- bundle adjustment
// poses: nKF x 16 float32 (Tcw row-major, in/out); points: nMP x 3 float32 (in/out); edges: mp, kf, kp xy, invSigma2.
// pose_out64: nKF x 7 (tx,ty,tz,qx,qy,qz,qw) fp64 state before the float32 cast; pts_out64: nMP x 3.
// log: up to logCap rows of (chi2, lambda, trials, accepted). Returns the number of LM iterations run.
int orc_local_ba(int nKF, int nMP, int nE, float* Tcw, const uint8_t* kfFixed, float* pts, const int* eMP, const int* eKF, const float* kpxy,
                 const float* invSigma2, int faceW, int faceH, const uint8_t* stopFlag, int its1, int its2, uint8_t* outlier,
                 double* pose_out64, double* pts_out64, double* log, int logCap) {
    LocalBA ba; ba.nKF = nKF; ba.nMP = nMP; ba.nE = nE; ba.W = faceW; ba.H = faceH; ba.f = faceW / 2.0;
    ba.pose.resize(nKF); ba.fixed.assign(kfFixed, kfFixed + nKF);
    for (int k = 0; k < nKF; k++) ba.pose[k] = se3_from_Tcw32(Tcw + 16 * k);
    ba.X.resize((size_t)nMP * 3); for (size_t i = 0; i < (size_t)nMP * 3; i++) ba.X[i] = (double)pts[i];
    ba.eMP.assign(eMP, eMP + nE); ba.eKF.assign(eKF, eKF + nE); ba.obs.resize(nE);
    for (int e = 0; e < nE; e++) ba.obs[e] = make_obs(kpxy[2 * e], kpxy[2 * e + 1], invSigma2[e], faceW, faceH);
    ba.stopFlag = stopFlag;
    ba.run(outlier, its1, its2);
    for (int k = 0; k < nKF; k++) {
        se3_to_Tcw32(ba.pose[k], Tcw + 16 * k);
        if (pose_out64) { double* o = pose_out64 + 7 * k; o[0] = ba.pose[k].t[0]; o[1] = ba.pose[k].t[1]; o[2] = ba.pose[k].t[2];
            o[3] = ba.pose[k].r.x; o[4] = ba.pose[k].r.y; o[5] = ba.pose[k].r.z; o[6] = ba.pose[k].r.w; }
    }
    for (size_t i = 0; i < (size_t)nMP * 3; i++) { pts[i] = (float)ba.X[i]; if (pts_out64) pts_out64[i] = ba.X[i]; }
    int n = (int)ba.log.size();
    for (int i = 0; i < n && i < logCap; i++) { log[4 * i] = ba.log[i].chi2; log[4 * i + 1] = ba.log[i].lambda; log[4 * i + 2] = ba.log[i].trials; log[4 * i + 3] = ba.log[i].accepted; }
    return n;
}
int orc_pose_opt(int n, float* Tcw, const float* Xw, const float* kpxy, const float* invSigma2, int faceW, int faceH, uint8_t* outlier,
                 double* pose_out64, double* log, int logCap, int* nIters) {
    PoseOpt po; po.n = n; po.W = faceW; po.H = faceH; po.f = faceW / 2.0;
    po.pose0 = se3_from_Tcw32(Tcw); po.Xw.resize((size_t)n * 3); po.obs.resize(n);
    for (int e = 0; e < n; e++) { for (int i = 0; i < 3; i++) po.Xw[3 * e + i] = (double)Xw[3 * e + i]; po.obs[e] = make_obs(kpxy[2 * e], kpxy[2 * e + 1], invSigma2[e], faceW, faceH); }
    int inl = po.run(outlier);
    if (n >= 3) se3_to_Tcw32(po.pose, Tcw);   // src/Optimizer.cpp:133-134 returns before SetPose
    if (pose_out64) { pose_out64[0] = po.pose.t[0]; pose_out64[1] = po.pose.t[1]; pose_out64[2] = po.pose.t[2];
        pose_out64[3] = po.pose.r.x; pose_out64[4] = po.pose.r.y; pose_out64[5] = po.pose.r.z; pose_out64[6] = po.pose.r.w; }
    int m = (int)po.log.size();
    for (int i = 0; i < m && i < logCap; i++) { log[4 * i] = po.log[i].chi2; log[4 * i + 1] = po.log[i].lambda; log[4 * i + 2] = po.log[i].trials; log[4 * i + 3] = po.log[i].accepted; }
    if (nIters) *nIters = m;
    return inl;
}
// exposed pieces for unit tests
// the reduced-camera-system solve of orc_local_ba: LDL^T without pivoting of the n x n row-major A (lower triangle read). 0 = zero / non-finite pivot.
int orc_ldlt_solve(const double* A, int n, const double* b, double* x) { return ldlt_solve(std::vector<double>(A, A + (size_t)n * n), n, b, x, false) ? 1 : 0; }
void orc_se3_exp(const double* u, double* out7) { SE3 s = se3_exp(u); out7[0] = s.t[0]; out7[1] = s.t[1]; out7[2] = s.t[2]; out7[3] = s.r.x; out7[4] = s.r.y; out7[5] = s.r.z; out7[6] = s.r.w; }
void orc_edge_eval(const float* Tcw, const double* X, float kx, float ky, int faceW, int faceH, double* err2, double* Jp12, double* Jx6, int* face) {
    SE3 T = se3_from_Tcw32(Tcw); EdgeObs o = make_obs(kx, ky, 1.f, faceW, faceH); double Xc[3], R[3][3], Jp[2][6], Jx[2][3];
    se3_map(T, X, Xc); quat_to_matrix(T.r, R); edge_error(o, faceW / 2.0, Xc, err2); edge_jacobians(o.face, faceW / 2.0, Xc, R, Jp, Jx);
    std::memcpy(Jp12, Jp, sizeof(Jp)); std::memcpy(Jx6, Jx, sizeof(Jx)); *face = o.face;
}
}
