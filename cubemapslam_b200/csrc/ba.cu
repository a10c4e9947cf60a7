// Optimizer::LocalBundleAdjustment of libcubemap_b200.so on sm_100a (PoseOptimization lives in pose_opt.cu).
//
// Reference (CPU, g2o): src/Optimizer.cpp:192-451; edge src/g2o_cubemap_vertices_edges.cpp:164-233; LM loop
// ThirdParty/g2o/g2o/core/optimization_algorithm_levenberg.cpp:61-189; Schur solve core/block_solver.hpp:354-486.
// The hypergraph is replaced by flat fp64 arrays; all arithmetic stays fp64 (the gate is 1e-5 relative on poses/points),
// including the reference's float32 round trip inside the projection (ba_math.cuh).
//
// Every accumulation is OUTPUT-STATIONARY (no floating-point atomics anywhere), hence bit-reproducible run to run:
//   k_ba_errors      per edge; chi2 by fixed-shape block sums + a last-block pass over the block partials
//   k_ba_lin_points  thread per landmark: Hll, bl in registers over the landmark's edges (sorted edge order), Hpl per edge
//   k_ba_lin_poses   CTA per free pose over its edge list: the 21+6 unique entries of (Hpp, bp)
//   k_ba_dinv        per landmark (Hll + lambda I)^-1 and Dinv*bl
//   k_ba_schur       CTA per pose pair (p1 <= p2) over the pair's precomputed co-observation list (edge a1 of p1, edge a2 of p2,
//                    same landmark, landmark order): S[p1,p2] = [p1==p2] Hpp - sum (B1 Dinv) B2^T, g[p1] = bp - sum B1 (Dinv bl)
//   k_ba_solve       one thread-block CLUSTER: blocked right-looking LDL^T of the n x n reduced camera system (n = 6 x free poses)
//                    with the right-hand side carried as an extra row; panel factorisation and trailing update spread over
//                    the cluster's SMs, panels exchanged through L2, cluster barriers between phases; no size cap
//   k_ba_backsub / k_ba_update / k_ba_scale / k_ba_restore   landmark back-substitution, oplus (with backup), gain-ratio scale
// Multi-GPU: landmarks (with their edges) are sharded l % nranks; every rank forms its partial [S | g | bpr | chi2 | scale]
// and the partials are summed either by one ncclAllReduce or by the one-shot NVLink kernel k_ba_xchg_reduce (peer pointers),
// in fixed rank order so that every rank solves bit-identical systems. Payloads are double-buffered by epoch parity: a rank may run one
// exchange ahead of a peer that is still reading the previous one.
// LM control flow (accept/reject, lambda schedule, ORB-SLAM2's stop rule, pbStopFlag) stays on the host like in the reference.
#include <cooperative_groups.h>
#include <dlfcn.h>
#include <algorithm>
#include <cfloat>
#include <chrono>
#include <cstring>
#include <vector>
#include "optimizer.cuh"

namespace cg = cooperative_groups;

namespace cslam {

struct BADev {
    int nKF, nMP, nE, nQ, nP, n;     // nQ non-fixed key frames (static per call), nP active free poses, n = 6 nP
    double f;                        // fx=fy=cx=cy
    Pose* pose; Pose* poseBak;
    double* X; double* Xbak;
    const int* eMP; const int* eKF;  // edges sorted by landmark (stable)
    const double* obs;               // 3 per edge: mx, my, w
    const int8_t* face;
    double* err; uint8_t* level;
    const int* poseIdx; const uint8_t* ptAct;   // per KF: compact active-free index or -1; per MP: 1 if it has an active edge
    const int* kfOfQ;                // per candidate pose q: KF index
    const int* lmStart;              // nMP+1, CSR over sorted edges
    const int* peStart; const int* peList;      // CSR of sorted edge ids by KF (ascending = landmark order)
    const long long* pairStart;      // nQ*nQ+1: co-observation list of (q1,q2), q1<=q2, row-major
    const int4* tuples;              // (a1, a2, landmark, -): the landmark rides along so that k_ba_schur has no tuple -> edge -> landmark load chain
    double *Hpp, *bp, *Hll, *bl, *Hpl, *Dinv, *db, *xp, *xl;
    double *S, *g, *bpr, *tail;      // one contiguous exchange buffer: [S n*n | g n | bpr n | tail 4]; tail = chi2, scale, -, -
    double* scal;                    // [0] chi2, [1] scale, [2] max diag (as bits), [3] solve flag, [4] lambda of the current trial
    double* part; unsigned* ticket;  // block partials + arrival counter of the deterministic grid reductions
    double* posePart; unsigned* poseTicket;   // k_ba_lin_poses: slice sums [nQ][POSE_SPLIT][27] + arrival counter per pose
    int robust; double delta, dsqr;
    int rank, nranks;                // landmark l is owned by rank l % nranks
};

static const int DINV_LD = 10;   // doubles per landmark in Dinv: 9 + 1 pad, so that every block is 16-byte aligned for the 128-bit loads of k_ba_schur

__device__ __forceinline__ bool owned(const BADev& D, int l) { return D.nranks == 1 || (l % D.nranks) == D.rank; }

// Deterministic grid-wide sum: fixed-shape block sums, block partials in part[], the last block to arrive adds them in a fixed shape.
// Returns true in thread 0 of the last block, with the total in *total.
__device__ __forceinline__ bool grid_sum(double v, double* part, unsigned* ticket, double* sh, double* total) {
    __shared__ bool last;
    const double s = block_sum(v, sh);
    if (threadIdx.x == 0) {
        part[blockIdx.x] = s;
        __threadfence();
        last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!last) return false;
    __threadfence();
    double t = 0;
    for (unsigned i = threadIdx.x; i < gridDim.x; i += blockDim.x) t += __ldcg(part + i);
    t = block_sum(t, sh);
    if (threadIdx.x == 0) { *total = t; *ticket = 0; }
    return threadIdx.x == 0;
}

// computeActiveErrors + activeRobustChi2 (partial sum over the landmarks this rank owns) -> *out
__global__ void __launch_bounds__(256) k_ba_errors(BADev D, double* out) {
    __shared__ double sh[32];
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    double c = 0;
    if (e < D.nE && D.level[e] == 0 && owned(D, D.eMP[e])) {
        double Xc[3], er[2];
        pose_map(D.pose[D.eKF[e]], D.X + 3 * D.eMP[e], Xc);
        edge_error(D.face[e], D.f, D.obs[3 * e], D.obs[3 * e + 1], Xc, er);
        D.err[2 * e] = er[0]; D.err[2 * e + 1] = er[1];
        const double chi = D.obs[3 * e + 2] * (er[0] * er[0] + er[1] * er[1]);
        if (D.robust) { double r0, r1; huber(D.delta, D.dsqr, chi, r0, r1); c = r0; } else c = chi;
    }
    double tot;
    if (grid_sum(c, D.part, D.ticket, sh, &tot)) *out = tot;
}

// Jacobians of one active edge (src/g2o_cubemap_vertices_edges.cpp:164-223) and its robust weight / weighted residual
struct EdgeLin { double Jx[2][3], Jp[2][6], w, r0, r1; };
__device__ __forceinline__ void linearize_edge(const BADev& D, int e, bool needPose, EdgeLin& L) {
    const int k = D.eKF[e], l = D.eMP[e];
    const Pose T = D.pose[k];
    double Xc[3], G[2][3], R[3][3];
    pose_map(T, D.X + 3 * l, Xc);
    edge_G(D.face[e], D.f, Xc, G);
    quat_to_matrix(T.q, R);
#pragma unroll
    for (int i = 0; i < 2; i++)
#pragma unroll
        for (int j = 0; j < 3; j++) L.Jx[i][j] = G[i][0] * R[0][j] + G[i][1] * R[1][j] + G[i][2] * R[2][j];
    if (needPose) edge_Jpose(G, Xc, L.Jp);
    const double e0 = D.err[2 * e], e1 = D.err[2 * e + 1], w0 = D.obs[3 * e + 2];
    double rho1 = 1.0;
    if (D.robust) { double r0; huber(D.delta, D.dsqr, w0 * (e0 * e0 + e1 * e1), r0, rho1); }
    L.w = rho1 * w0; L.r0 = -L.w * e0; L.r1 = -L.w * e1;
}

// buildSystem, landmark side (base_binary_edge.hpp:55-120): Hll, bl of one landmark accumulated in registers in edge order, Hpl per edge
static const int LM_LANES = 4;   // lanes that share one landmark in k_ba_lin_points / k_ba_backsub (edge a of the landmark goes to lane a % 4)
__global__ void __launch_bounds__(128) k_ba_lin_points(BADev D) {
    const int l = (blockIdx.x * blockDim.x + threadIdx.x) / LM_LANES, sub = threadIdx.x % LM_LANES;
    const bool mine = l < D.nMP && owned(D, l);
    double H[6] = {0, 0, 0, 0, 0, 0}, b[3] = {0, 0, 0};
    const int eBeg = mine ? D.lmStart[l] : 0, eEnd = mine ? D.lmStart[l + 1] : 0;
    for (int e = eBeg + sub; e < eEnd; e += LM_LANES) {
        double* B = D.Hpl + 18 * (size_t)e;
        const int pi = D.poseIdx[D.eKF[e]];
        if (D.level[e] != 0) {   // inactive edges contribute zero blocks (the co-observation lists are built once per call)
#pragma unroll
            for (int i = 0; i < 18; i++) B[i] = 0.0;
            continue;
        }
        EdgeLin L;
        linearize_edge(D, e, pi >= 0, L);
        int q = 0;
#pragma unroll
        for (int i = 0; i < 3; i++) {
            b[i] += L.Jx[0][i] * L.r0 + L.Jx[1][i] * L.r1;
#pragma unroll
            for (int j = i; j < 3; j++) H[q++] += L.w * (L.Jx[0][i] * L.Jx[0][j] + L.Jx[1][i] * L.Jx[1][j]);
        }
        if (pi >= 0) {
#pragma unroll
            for (int i = 0; i < 6; i++)
#pragma unroll
                for (int j = 0; j < 3; j++) B[3 * i + j] = L.w * (L.Jp[0][i] * L.Jx[0][j] + L.Jp[1][i] * L.Jx[1][j]);
        } else {
#pragma unroll
            for (int i = 0; i < 18; i++) B[i] = 0.0;
        }
    }
    // fixed-shape sum over the 4 lanes of the landmark (all 32 lanes of the warp take part)
#pragma unroll
    for (int i = 0; i < 6; i++) { H[i] += __shfl_xor_sync(0xffffffffu, H[i], 1); H[i] += __shfl_xor_sync(0xffffffffu, H[i], 2); }
#pragma unroll
    for (int i = 0; i < 3; i++) { b[i] += __shfl_xor_sync(0xffffffffu, b[i], 1); b[i] += __shfl_xor_sync(0xffffffffu, b[i], 2); }
    if (!mine || sub) return;
    double* Hl = D.Hll + 9 * (size_t)l;
    Hl[0] = H[0]; Hl[1] = H[1]; Hl[2] = H[2]; Hl[3] = H[1]; Hl[4] = H[3]; Hl[5] = H[4]; Hl[6] = H[2]; Hl[7] = H[4]; Hl[8] = H[5];
    D.bl[3 * l] = b[0]; D.bl[3 * l + 1] = b[1]; D.bl[3 * l + 2] = b[2];
}

// buildSystem, pose side: POSE_SPLIT CTAs per candidate pose, each over a slice of the pose's edge list; 21 unique entries of Hpp + 6 of bp.
// Slice sums go to posePart[q][slice][27]; the last CTA of the pose to arrive adds the slices in slice order (fixed shape -> reproducible).
static const int POSE_SPLIT = 8;
__global__ void __launch_bounds__(256) k_ba_lin_poses(BADev D) {
    __shared__ double red[8][28];
    __shared__ bool last;
    const int qi = blockIdx.x, sl = blockIdx.y;
    const int k = D.kfOfQ[qi], p = D.poseIdx[k];
    if (p < 0) return;
    double acc[27];
#pragma unroll
    for (int i = 0; i < 27; i++) acc[i] = 0.0;
    for (int q = D.peStart[k] + sl * 256 + threadIdx.x; q < D.peStart[k + 1]; q += POSE_SPLIT * 256) {
        const int e = D.peList[q];
        if (D.level[e] != 0 || !owned(D, D.eMP[e])) continue;
        EdgeLin L;
        linearize_edge(D, e, true, L);
        int t = 0;
#pragma unroll
        for (int a = 0; a < 6; a++)
#pragma unroll
            for (int b = a; b < 6; b++) acc[t++] += L.w * (L.Jp[0][a] * L.Jp[0][b] + L.Jp[1][a] * L.Jp[1][b]);
#pragma unroll
        for (int a = 0; a < 6; a++) acc[21 + a] += L.Jp[0][a] * L.r0 + L.Jp[1][a] * L.r1;
    }
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < 27; i++) {
        double v = acc[i];
#pragma unroll
        for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) red[w][i] = v;
    }
    __syncthreads();
    double* mine = D.posePart + ((size_t)qi * POSE_SPLIT + sl) * 27;
    if (threadIdx.x < 27) {
        double s = 0;
        for (int ww = 0; ww < 8; ww++) s += red[ww][threadIdx.x];
        __stcg(mine + threadIdx.x, s);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(D.poseTicket + qi, 1u) == POSE_SPLIT - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    if (threadIdx.x < 27) {
        double s = 0;
        for (int j = 0; j < POSE_SPLIT; j++) s += __ldcg(D.posePart + ((size_t)qi * POSE_SPLIT + j) * 27 + threadIdx.x);
        red[0][threadIdx.x] = s;
    }
    if (threadIdx.x == 0) D.poseTicket[qi] = 0;
    __syncthreads();
    if (threadIdx.x < 36) {
        const int a = threadIdx.x / 6, b = threadIdx.x % 6, lo = min(a, b), hi = max(a, b);
        D.Hpp[36 * p + threadIdx.x] = red[0][lo * 6 - lo * (lo - 1) / 2 + (hi - lo)];
    }
    if (threadIdx.x < 6) D.bp[6 * p + threadIdx.x] = red[0][21 + threadIdx.x];
}

// computeLambdaInit: max |H_jj| over all active free vertices (integer atomicMax of the bit pattern: order independent)
__global__ void __launch_bounds__(256) k_ba_maxdiag(BADev D) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    double m = 0;
    if (i < D.nP * 6) m = fabs(D.Hpp[36 * (i / 6) + 7 * (i % 6)]);
    const int j = i - D.nP * 6;
    if (j >= 0 && j < D.nMP * 3) { const int l = j / 3; if (D.ptAct[l] && owned(D, l)) m = fabs(D.Hll[9 * l + 4 * (j % 3)]); }
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(reinterpret_cast<unsigned long long*>(&D.scal[2]), (unsigned long long)__double_as_longlong(m));
}

// Dinv = (Hll + lambda I)^-1 (3x3 cofactors, like Eigen), db = Dinv * bl
__global__ void __launch_bounds__(256) k_ba_dinv(BADev D) {
    const double lambda = D.scal[4];
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= D.nMP || !owned(D, l)) return;
    double* Dv = D.Dinv + DINV_LD * (size_t)l;
    if (!D.ptAct[l]) {
#pragma unroll
        for (int i = 0; i < 9; i++) Dv[i] = 0.0;
        D.db[3 * l] = 0; D.db[3 * l + 1] = 0; D.db[3 * l + 2] = 0;
        return;
    }
    double M[9];
#pragma unroll
    for (int i = 0; i < 9; i++) M[i] = D.Hll[9 * (size_t)l + i];
    M[0] += lambda; M[4] += lambda; M[8] += lambda;
    const double c00 = M[4] * M[8] - M[5] * M[7], c01 = M[5] * M[6] - M[3] * M[8], c02 = M[3] * M[7] - M[4] * M[6];
    const double id = 1.0 / (M[0] * c00 + M[1] * c01 + M[2] * c02);
    double Di[9];
    Di[0] = c00 * id; Di[1] = (M[2] * M[7] - M[1] * M[8]) * id; Di[2] = (M[1] * M[5] - M[2] * M[4]) * id;
    Di[3] = c01 * id; Di[4] = (M[0] * M[8] - M[2] * M[6]) * id; Di[5] = (M[2] * M[3] - M[0] * M[5]) * id;
    Di[6] = c02 * id; Di[7] = (M[1] * M[6] - M[0] * M[7]) * id; Di[8] = (M[0] * M[4] - M[1] * M[3]) * id;
#pragma unroll
    for (int i = 0; i < 9; i++) Dv[i] = Di[i];
#pragma unroll
    for (int i = 0; i < 3; i++) D.db[3 * l + i] = Di[3 * i] * D.bl[3 * l] + Di[3 * i + 1] * D.bl[3 * l + 1] + Di[3 * i + 2] * D.bl[3 * l + 2];
}

// ---- co-observation lists: for every pair of candidate poses q1 <= q2 the (a1, a2) edge pairs that share a landmark, in landmark order.
// Built once per cslam_local_ba call over ALL edges (edges that become inactive later carry zero Hpl blocks).
__device__ __forceinline__ int partner_edge(const BADev& D, int a1, int k2) {
    const int l = D.eMP[a1];
    for (int a2 = D.lmStart[l]; a2 < D.lmStart[l + 1]; a2++) if (D.eKF[a2] == k2) return a2;
    return -1;
}
__global__ void __launch_bounds__(128) k_ba_pairs_count(BADev D, long long* cnt) {
    __shared__ int wsum[4];
    const int q1 = blockIdx.y, q2 = blockIdx.x;
    if (q1 > q2) { if (threadIdx.x == 0) cnt[(size_t)q1 * D.nQ + q2] = 0; return; }
    const int k1 = D.kfOfQ[q1], k2 = D.kfOfQ[q2], beg = D.peStart[k1], end = D.peStart[k1 + 1];
    if (q1 == q2) { if (threadIdx.x == 0) cnt[(size_t)q1 * D.nQ + q2] = end - beg; return; }
    int c = 0;
    for (int q = beg + threadIdx.x; q < end; q += blockDim.x) c += partner_edge(D, D.peList[q], k2) >= 0;
#pragma unroll
    for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) cnt[(size_t)q1 * D.nQ + q2] = wsum[0] + wsum[1] + wsum[2] + wsum[3];
}
// exclusive scan of `m` counts (in place) + total, one CTA
__global__ void __launch_bounds__(1024) k_ba_pairs_scan(long long* v, int m) {
    __shared__ long long wtot[32];
    __shared__ long long carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int base = 0; base < m; base += 1024) {
        const int i = base + threadIdx.x;
        const long long x = i < m ? v[i] : 0;
        long long s = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const long long t = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += t; }
        if (lane == 31) wtot[w] = s;
        __syncthreads();
        if (w == 0) {
            long long t = wtot[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const long long u = __shfl_up_sync(0xffffffffu, t, o); if (lane >= o) t += u; }
            wtot[lane] = t;
        }
        __syncthreads();
        const long long excl = carry + (w ? wtot[w - 1] : 0) + s - x;
        if (i < m) v[i] = excl;
        __syncthreads();
        if (threadIdx.x == 1023) carry = excl + x;
        __syncthreads();
    }
    if (threadIdx.x == 0) v[m] = carry;
}
__global__ void __launch_bounds__(128) k_ba_pairs_fill(BADev D, const long long* start, int4* tuples) {
    __shared__ int wcnt[4];
    __shared__ long long base;
    const int q1 = blockIdx.y, q2 = blockIdx.x;
    if (q1 > q2) return;
    const int k1 = D.kfOfQ[q1], k2 = D.kfOfQ[q2], beg = D.peStart[k1], end = D.peStart[k1 + 1];
    int4* out = tuples + start[(size_t)q1 * D.nQ + q2];
    if (q1 == q2) { for (int q = beg + threadIdx.x; q < end; q += blockDim.x) { const int a = D.peList[q]; out[q - beg] = make_int4(a, a, D.eMP[a], 0); } return; }
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int q0 = beg; q0 < end; q0 += blockDim.x) {   // ordered compaction: output order = order of the pose's edge list = landmark order
        const int q = q0 + threadIdx.x;
        int a1 = -1, a2 = -1;
        if (q < end) { a1 = D.peList[q]; a2 = partner_edge(D, a1, k2); }
        const unsigned ball = __ballot_sync(0xffffffffu, a2 >= 0);
        if (lane == 0) wcnt[w] = __popc(ball);
        __syncthreads();
        int pre = 0;
        for (int ww = 0; ww < w; ww++) pre += wcnt[ww];
        if (a2 >= 0) out[base + pre + __popc(ball & ((1u << lane) - 1))] = make_int4(a1, a2, D.eMP[a1], 0);
        __syncthreads();
        if (threadIdx.x == 0) base += wcnt[0] + wcnt[1] + wcnt[2] + wcnt[3];
        __syncthreads();
    }
}

// Schur complement (block_solver.hpp:381-439), output-stationary: one CTA per pose pair accumulates its 6x6 block in registers over the
// pair's co-observation list, then a fixed-shape reduction. The diagonal pair also forms g = bp - sum B (Dinv bl) and bpr = bp.
// Two threads share a tuple (rows 0-2 / rows 3-5 of the 6x6 block): 18 + 3 accumulators per thread keep the kernel at a register count
// that lets the list loads of many tuples be in flight per SM (the kernel is L2-latency bound, the Hpl / Dinv blocks are L2 resident).
static const int SCHUR_T = 256;
__global__ void __launch_bounds__(SCHUR_T) k_ba_schur(BADev D, int addLambda) {
    const double lambdaDiag = addLambda ? D.scal[4] : 0.0;
    __shared__ double red[SCHUR_T / 32][44];
    const int q1 = blockIdx.y, q2 = blockIdx.x;
    if (q1 > q2) return;
    const int p1 = D.poseIdx[D.kfOfQ[q1]], p2 = D.poseIdx[D.kfOfQ[q2]];
    if (p1 < 0 || p2 < 0) return;
    const bool diag = q1 == q2;
    const int h = threadIdx.x & 1;
    double acc[21];
#pragma unroll
    for (int i = 0; i < 21; i++) acc[i] = 0.0;
    const long long beg = D.pairStart[(size_t)q1 * D.nQ + q2], end = D.pairStart[(size_t)q1 * D.nQ + q2 + 1];
    long long t = beg + (threadIdx.x >> 1);
    int4 nxt = t < end ? D.tuples[t] : make_int4(0, 0, 0, 0);
    for (; t < end; t += SCHUR_T / 2) {
        const int4 tp = nxt;
        if (t + SCHUR_T / 2 < end) nxt = D.tuples[t + SCHUR_T / 2];   // the next tuple's index load flies under this tuple's block loads
        const int l = tp.z;
        if (!owned(D, l)) continue;
        // 19 128-bit loads per thread: every lane reads a different block, so the L1 wavefront count per byte is what bounds this kernel
        const double2* B1v = reinterpret_cast<const double2*>(D.Hpl + 18 * (size_t)tp.x) + 4 * h;   // doubles 8h .. 8h+9: rows 3h..3h+2 are w[h .. h+8]
        const double2* B2v = reinterpret_cast<const double2*>(D.Hpl + 18 * (size_t)tp.y);
        const double2* Div = reinterpret_cast<const double2*>(D.Dinv + DINV_LD * (size_t)l);
        double w[10], di[10], b2[18], b1[9];
#pragma unroll
        for (int i = 0; i < 5; i++) { const double2 v = B1v[i]; w[2 * i] = v.x; w[2 * i + 1] = v.y; const double2 u = Div[i]; di[2 * i] = u.x; di[2 * i + 1] = u.y; }
#pragma unroll
        for (int i = 0; i < 9; i++) { const double2 v = B2v[i]; b2[2 * i] = v.x; b2[2 * i + 1] = v.y; }
#pragma unroll
        for (int i = 0; i < 9; i++) b1[i] = h ? w[i + 1] : w[i];
#pragma unroll
        for (int i = 0; i < 3; i++) {
            const double t0 = b1[3 * i] * di[0] + b1[3 * i + 1] * di[3] + b1[3 * i + 2] * di[6];
            const double t1 = b1[3 * i] * di[1] + b1[3 * i + 1] * di[4] + b1[3 * i + 2] * di[7];
            const double t2 = b1[3 * i] * di[2] + b1[3 * i + 1] * di[5] + b1[3 * i + 2] * di[8];
#pragma unroll
            for (int j = 0; j < 6; j++) acc[6 * i + j] += t0 * b2[3 * j] + t1 * b2[3 * j + 1] + t2 * b2[3 * j + 2];
        }
        if (diag) {
            const double d0 = D.db[3 * l], d1 = D.db[3 * l + 1], d2 = D.db[3 * l + 2];
#pragma unroll
            for (int i = 0; i < 3; i++) acc[18 + i] += b1[3 * i] * d0 + b1[3 * i + 1] * d1 + b1[3 * i + 2] * d2;
        }
    }
    // lanes of equal parity hold the same rows: xor offsets 16 .. 2 leave the row sums in lanes 0 (rows 0-2) and 1 (rows 3-5)
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < 21; i++) {
        if (i >= 18 && !diag) break;
        double v = acc[i];
#pragma unroll
        for (int o = 16; o > 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane < 2) red[w][i < 18 ? 18 * lane + i : 36 + 3 * lane + (i - 18)] = v;
    }
    __syncthreads();
    const int n = D.n;
    if (threadIdx.x < 36) {
        const int i = threadIdx.x / 6, j = threadIdx.x % 6;
        double s = 0;
#pragma unroll
        for (int ww = 0; ww < SCHUR_T / 32; ww++) s += red[ww][threadIdx.x];
        double v = -s;
        if (diag) { v += D.Hpp[36 * p1 + threadIdx.x]; if (i == j) v += lambdaDiag; }
        D.S[(size_t)(6 * p1 + i) * n + 6 * p2 + j] = v;
        if (!diag) D.S[(size_t)(6 * p2 + j) * n + 6 * p1 + i] = v;
    } else if (diag && threadIdx.x < 42) {
        const int i = threadIdx.x - 36;
        double s = 0;
#pragma unroll
        for (int ww = 0; ww < SCHUR_T / 32; ww++) s += red[ww][threadIdx.x];
        const double b = D.bp[6 * p1 + i];
        D.g[6 * p1 + i] = b - s;
        D.bpr[6 * p1 + i] = b;
    }
}

// ---------------------------------------------------------------------------------------------- reduced camera system solve
// Blocked right-looking LDL^T (no pivoting; LinearSolverEigen's SimplicialLDLT has none either) of the n x n system in ONE thread-block
// cluster. The right-hand side g sits right behind S, i.e. it is row n of an (n+1) x n matrix: carrying it through the factorisation
// as one more row performs the forward substitution (row n of L = D^-1 L^-1 g).
//
// Everything here is LATENCY bound (n ~ 300: 9 MFLOP; measured on B200, tools/ubench_fp64.cu: DFMA 8 clk, fp64 divide 127 clk, shared
// load 29 clk, __syncthreads 38 clk, L2 load 375 clk, cluster barrier 420 clk), so every phase is written to keep its dependent chain short
// and to have all of a thread's L2 loads in flight together. Per panel of NB = 32 columns:
//   (1) every CTA factors the NB x NB diagonal block redundantly: thread (r, g) keeps elements (r, 4g..4g+3) in registers, the pivot column is
//       published through a double-buffered shared column -> one barrier per column; 1 / pivot = rcp.approx + 2 Newton steps (~55 clk).
//       Then M = (unit lower factor)^-1: each warp solves L m = e_k for 4 columns, lane = row, pivot entries by shuffle (no barrier);
//   (2) the rows below become a product instead of forward substitutions: X = A_rows M^T, L = X / d; FOUR lanes per row, lane j forms
//       the columns j, j+4, ... from the row held in registers (no dependent chain, no shuffles), a contiguous chunk of rows per CTA;
//       L goes back into S (row-major, for the back substitution) and L, L d go to the transposed panel buffers Lt / LDt;
//   (3) cluster barrier; every CTA copies both panels to shared memory (16-byte L2 loads, 4 in flight per thread); trailing update with
//       4 x 2 register tiles enumerated over the lower triangle only and dealt over all threads of the cluster; cluster barrier.
// Back substitution by cluster rank 0, panel by panel from the bottom: x_b = M_b^T y_b (one warp, 32 independent products per lane; M_b
// was parked in L2 scratch by (2)) instead of a 32-step triangular solve, then the rows above take y -= L_b^T x_b. scal[3] = 1 on a zero / non-finite pivot (LinearSolverEigen's failure): the LM trial is rejected.
static const int LD_NB = 32;
static const int SOLVE_T = 256;

// 1 / d to within an ulp: MUFU.RCP64H seed (~20 bits) and two Newton steps, instead of the ~127 clk IEEE divide on the critical path
__device__ __forceinline__ double fast_rcp(double d) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
    r = fma(r, fma(-d, r, 1.0), r);
    r = fma(r, fma(-d, r, 1.0), r);
    return r;
}

__global__ void __launch_bounds__(SOLVE_T) k_ba_solve(BADev D, double* __restrict__ Lt, double* __restrict__ LDt, double* __restrict__ Mg, int ldp, int stage, long long* prof) {
    extern __shared__ double dsm[];                 // [stage ? 2 * NB * ldp : 0] panels, then y[n] for the back substitution
    __shared__ double Pd[LD_NB][LD_NB + 1];         // L of the diagonal block (strictly lower part)
    __shared__ double Msm[LD_NB][LD_NB + 1];        // M = L^-1 of the diagonal block (zeros above the diagonal)
    __shared__ double colbuf[2][LD_NB];             // the pivot column of the current / next step
    __shared__ double dinvv[LD_NB];
    __shared__ int fail;
    cg::cluster_group cluster = cg::this_cluster();
    const int C = cluster.num_blocks(), crank = cluster.block_rank();
    const int n = D.n, tid = threadIdx.x;
    double* A = D.S;
    double* sL = dsm; double* sLD = dsm + (size_t)LD_NB * ldp;
    if (tid == 0) fail = 0;
    __syncthreads();
    long long tprev = 0, tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const bool doProf = prof && crank == 0 && tid == 0;
#define SOLVE_MARK(k) do { if (doProf) { const long long tn = clock64(); tacc[k] += tn - tprev; tprev = tn; } } while (0)
    if (doProf) tprev = clock64();
    for (int jb = 0; jb < n; jb += LD_NB) {
        const int nb = min(LD_NB, n - jb), rows = n + 1 - jb;
        // (1) diagonal block: thread (r, g) owns (r, 4g .. 4g+3)
        const int r = tid >> 3, g4 = (tid & 7) * 4;
        double a[4];
#pragma unroll
        for (int k = 0; k < 4; k++) { const int c = g4 + k; a[k] = (r < nb && c <= r) ? __ldcg(A + (size_t)(jb + r) * n + jb + c) : 0.0; }
        if (g4 == 0) colbuf[0][r] = a[0];
        __syncthreads();
        SOLVE_MARK(0);
#pragma unroll
        for (int c = 0; c < LD_NB; c++) {
            if (c < nb) {   // block-uniform
                const double* col = colbuf[c & 1];
                const double dc = col[c], ld = col[r];
                double l4[4];
#pragma unroll
                for (int k = 0; k < 4; k++) l4[k] = col[g4 + k];
                const double inv = fast_rcp(dc);
                if (tid == 0) dinvv[c] = inv;
                if (r > c) {
#pragma unroll
                    for (int k = 0; k < 4; k++) { const int c2 = g4 + k; if (c2 > c && c2 <= r) a[k] -= ld * (l4[k] * inv); }
                }
                if ((c >> 2) == (tid & 7)) Pd[r][c] = r > c ? ld * inv : 0.0;
                if (c + 1 < nb && ((c + 1) >> 2) == (tid & 7)) colbuf[(c + 1) & 1][r] = a[(c + 1) & 3];
                __syncthreads();
            }
        }
        // M = L^-1: warp w solves L m = e_k for the columns k = w, w+8, w+16, w+24 (lane = row; right-looking, the pivot entry travels by shuffle,
        // no block barrier inside). Columns >= nb of a short last panel stay unit vectors and are never used.
        {
            const int w = tid >> 5, ln = tid & 31;
            double mk[4], lrow[LD_NB];
#pragma unroll
            for (int c = 0; c < LD_NB; c++) lrow[c] = (c < nb && ln < nb && ln > c) ? Pd[ln][c] : 0.0;
#pragma unroll
            for (int q = 0; q < 4; q++) mk[q] = ln == w + 8 * q ? 1.0 : 0.0;
#pragma unroll
            for (int c = 0; c < LD_NB; c++) {
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    if (c >= 8 * q) {   // column k = w + 8q is zero above row k >= 8q: earlier steps do nothing
                        const double mc = __shfl_sync(0xffffffffu, mk[q], c);
                        mk[q] -= lrow[c] * mc;   // lrow[c] == 0 for lanes <= c
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < 4; q++) Msm[ln][w + 8 * q] = mk[q];
        }
        __syncthreads();
        if (tid < nb) { const double iv = dinvv[tid]; if (!isfinite(iv) || iv == 0.0) fail = 1; }   // zero / non-finite pivot <=> its reciprocal is not a finite non-zero number
        __syncthreads();
        SOLVE_MARK(1);
        if (fail) break;   // block-uniform and identical in every CTA of the cluster (same data)
        // (2) rows below the diagonal block (including the rhs row): a contiguous chunk of rows per CTA, 4 lanes per row, 8 columns per lane.
        // Per element the subtractions run over c2 = 0, 1, ... in the order of the plain forward substitution.
        const int trR = rows - nb;
        const int chunk = (trR + C - 1) / C, r0c = crank * chunk, r1c = min(r0c + chunk, trR);
        {
            // X = A_rows M^T (x_c = sum_{c2 <= c} a_c2 M[c][c2]), L = X / d. 4 lanes per row; lane j forms the columns j, j+4, ... (balanced: the
            // sum for column j + 4 m runs to c2 = 4 m + 3, the entries of M above the diagonal are zeros) from the whole row held in registers.
            const int j = tid & 3, slot = tid >> 2;
            for (int base = r0c; base < r1c; base += SOLVE_T / 4) {
                const int rr = base + slot;
                const bool valid = rr < r1c;
                double* Arow = A + (size_t)(jb + nb + (valid ? rr : r0c)) * n + jb;
                double av[LD_NB];
#pragma unroll
                for (int c = 0; c < LD_NB; c++) av[c] = (valid && c < nb) ? __ldcg(Arow + c) : 0.0;
                const double* Mj = &Msm[j][0];
#pragma unroll
                for (int mq = 0; mq < LD_NB / 4; mq++) {
                    if (4 * mq < nb) {   // block-uniform
                        double x0 = 0, x1 = 0;
#pragma unroll
                        for (int c2 = 0; c2 < 4 * mq + 4; c2 += 2) { x0 += av[c2] * Mj[4 * mq * (LD_NB + 1) + c2]; x1 += av[c2 + 1] * Mj[4 * mq * (LD_NB + 1) + c2 + 1]; }
                        const double x = x0 + x1;
                        const int c = j + 4 * mq;
                        if (valid && c < nb) {
                            const double lv = x * dinvv[c];
                            __stcg(Arow + c, lv);
                            __stcg(Lt + (size_t)c * ldp + rr, lv); __stcg(LDt + (size_t)c * ldp + rr, x);
                        }
                    }
                }
            }
        }
        // M of this panel to the scratch the back substitution reads (cluster rank 0)
        if (crank == 0)
            for (int i = tid; i < LD_NB * LD_NB; i += SOLVE_T) { const int rr = i / LD_NB, c = i - rr * LD_NB; __stcg(Mg + (size_t)(jb / LD_NB) * LD_NB * LD_NB + i, (rr < nb && c < nb) ? Msm[rr][c] : 0.0); }
        SOLVE_MARK(2);
        cluster.sync();
        SOLVE_MARK(3);
        // (3) trailing update A[i][k] -= sum_c (L d)[i][c] L[k][c], rows i include the rhs row, columns k < trC, k <= i
        const int trC = n - jb - nb;
        if (trC > 0) {
            if (stage) {
                // thread (half, q): panel columns c = 2 u + half, double2 words q and q + 128 of a panel row; 8 columns (16 .. 32 loads) in flight
                const int w2 = (trR + 1) >> 1, st2 = ldp >> 1, half = tid >> 7, q0 = tid & 127;
                const double2* gL = reinterpret_cast<const double2*>(Lt); const double2* gD = reinterpret_cast<const double2*>(LDt);
                double2* hL = reinterpret_cast<double2*>(sL); double2* hD = reinterpret_cast<double2*>(sLD);
                const bool q0ok = q0 < w2, q1ok = q0 + 128 < w2;
                for (int c0 = half; c0 < nb; c0 += 16) {
                    double2 vl[8][2], vd[8][2];
#pragma unroll
                    for (int u = 0; u < 8; u++) {
                        const int c = c0 + 2 * u;
                        if (c < nb) {
                            if (q0ok) { vl[u][0] = __ldcg(gL + c * st2 + q0); vd[u][0] = __ldcg(gD + c * st2 + q0); }
                            if (q1ok) { vl[u][1] = __ldcg(gL + c * st2 + q0 + 128); vd[u][1] = __ldcg(gD + c * st2 + q0 + 128); }
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 8; u++) {
                        const int c = c0 + 2 * u;
                        if (c < nb) {
                            if (q0ok) { hL[c * st2 + q0] = vl[u][0]; hD[c * st2 + q0] = vd[u][0]; }
                            if (q1ok) { hL[c * st2 + q0 + 128] = vl[u][1]; hD[c * st2 + q0 + 128] = vd[u][1]; }
                        }
                    }
                }
                for (int q = q0 + 256; q < w2; q += 128)   // panels longer than 512 rows (not the staged regime in practice)
                    for (int c = half; c < nb; c += 2) { hL[c * st2 + q] = __ldcg(gL + c * st2 + q); hD[c * st2 + q] = __ldcg(gD + c * st2 + q); }
                __syncthreads();
            }
            SOLVE_MARK(4);
            const int tR = (trR + 3) >> 2, tC = (trC + 1) >> 1;
            // tile row br (4 rows) holds the tile columns bc with 2 bc <= 4 br + 3, i.e. bc <= 2 br + 1: 2 br + 2 tiles, br (br + 1) before it
            const int nTiles = tR * (tR + 1);
            for (int i = crank * SOLVE_T + tid; i < nTiles; i += C * SOLVE_T) {
                int br = (int)((sqrtf(4.0f * (float)i + 1.0f) - 1.0f) * 0.5f);
                while (br * (br + 1) > i) br--;
                while ((br + 1) * (br + 2) <= i) br++;
                const int bc = i - br * (br + 1);
                if (bc >= tC) continue;
                const int r0 = 4 * br, k0 = 2 * bc;
                // destination values first: their L2 latency runs under the product loop
                double dv[4][2]; bool ok[4][2];
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const int rr = r0 + q;
                    const double* dst = A + (size_t)(jb + nb + min(rr, trR - 1)) * n + jb + nb;
                    ok[q][0] = rr < trR && k0 <= rr && k0 < trC; ok[q][1] = rr < trR && k0 + 1 <= rr && k0 + 1 < trC;
                    dv[q][0] = ok[q][0] ? __ldcg(dst + k0) : 0.0; dv[q][1] = ok[q][1] ? __ldcg(dst + k0 + 1) : 0.0;
                }
                double acc[4][2] = {{0, 0}, {0, 0}, {0, 0}, {0, 0}};
                if (stage) {
                    const double2* qL = reinterpret_cast<const double2*>(sL + k0);
                    const double2* qD = reinterpret_cast<const double2*>(sLD + r0);
                    const int st = ldp >> 1;
#pragma unroll 8
                    for (int c = 0; c < nb; c++) {
                        const double2 bv = qL[c * st], a01 = qD[c * st], a23 = qD[c * st + 1];
                        acc[0][0] += a01.x * bv.x; acc[0][1] += a01.x * bv.y; acc[1][0] += a01.y * bv.x; acc[1][1] += a01.y * bv.y;
                        acc[2][0] += a23.x * bv.x; acc[2][1] += a23.x * bv.y; acc[3][0] += a23.y * bv.x; acc[3][1] += a23.y * bv.y;
                    }
                } else {
#pragma unroll 8
                    for (int c = 0; c < nb; c++) {
                        const double2 bv = __ldcg(reinterpret_cast<const double2*>(Lt + (size_t)c * ldp + k0));
                        const double2 a01 = __ldcg(reinterpret_cast<const double2*>(LDt + (size_t)c * ldp + r0));
                        const double2 a23 = __ldcg(reinterpret_cast<const double2*>(LDt + (size_t)c * ldp + r0 + 2));
                        acc[0][0] += a01.x * bv.x; acc[0][1] += a01.x * bv.y; acc[1][0] += a01.y * bv.x; acc[1][1] += a01.y * bv.y;
                        acc[2][0] += a23.x * bv.x; acc[2][1] += a23.x * bv.y; acc[3][0] += a23.y * bv.x; acc[3][1] += a23.y * bv.y;
                    }
                }
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    double* dst = A + (size_t)(jb + nb + min(r0 + q, trR - 1)) * n + jb + nb;
                    if (ok[q][0]) __stcg(dst + k0, dv[q][0] - acc[q][0]);
                    if (ok[q][1]) __stcg(dst + k0 + 1, dv[q][1] - acc[q][1]);
                }
            }
        }
        SOLVE_MARK(5);
        cluster.sync();
        SOLVE_MARK(6);
    }
    if (fail) { if (crank == 0 && tid == 0) D.scal[3] = 1.0; return; }
    if (crank != 0) return;
    // backward: L^T x = z, z = row n of L (= D^-1 L^-1 g), panel by panel from the bottom: x_b = M_b^T y_b, then y_above -= L[b][above]^T x_b
    double* y = dsm + (stage ? 2 * (size_t)LD_NB * ldp : 0);
    for (int i = tid; i < n; i += SOLVE_T) y[i] = __ldcg(A + (size_t)n * n + i);
    __syncthreads();
    for (int pb = (n - 1) / LD_NB; pb >= 0; pb--) {
        const int j0 = pb * LD_NB, nb = min(LD_NB, n - j0);
        // rows above the block: L[j0 + j][i] for this thread's rows i; M_b[j][lane] for warp 0 (all independent of y: in flight together)
        double v0[LD_NB], v1[LD_NB];
        const int i0 = tid, i1 = tid + SOLVE_T;
#pragma unroll
        for (int j = 0; j < LD_NB; j++) {
            v0[j] = (j < nb && i0 < j0) ? __ldcg(A + (size_t)(j0 + j) * n + i0) : 0.0;
            v1[j] = (j < nb && i1 < j0) ? __ldcg(A + (size_t)(j0 + j) * n + i1) : 0.0;
        }
        if (tid < 32) {
            double mc[LD_NB], yv[LD_NB];
#pragma unroll
            for (int j = 0; j < LD_NB; j++) { mc[j] = __ldcg(Mg + (size_t)pb * LD_NB * LD_NB + j * LD_NB + tid); yv[j] = j < nb ? y[j0 + j] : 0.0; }
            double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
#pragma unroll
            for (int j = 0; j < LD_NB; j += 4) { s0 += mc[j] * yv[j]; s1 += mc[j + 1] * yv[j + 1]; s2 += mc[j + 2] * yv[j + 2]; s3 += mc[j + 3] * yv[j + 3]; }
            __syncwarp();
            if (tid < nb) y[j0 + tid] = (s0 + s1) + (s2 + s3);
        }
        __syncthreads();
        {
            double s0 = 0, s1 = 0;
#pragma unroll
            for (int j = 0; j < LD_NB; j++) if (j < nb) { const double xj = y[j0 + j]; s0 += v0[j] * xj; s1 += v1[j] * xj; }
            if (i0 < j0) y[i0] -= s0;
            if (i1 < j0) y[i1] -= s1;
        }
        for (int i = tid + 2 * SOLVE_T; i < j0; i += SOLVE_T) {
            double sacc = 0;
            for (int j = 0; j < nb; j++) sacc += __ldcg(A + (size_t)(j0 + j) * n + i) * y[j0 + j];
            y[i] -= sacc;
        }
        __syncthreads();
    }
    for (int i = tid; i < n; i += SOLVE_T) D.xp[i] = y[i];
    SOLVE_MARK(7);
    if (doProf) for (int k = 0; k < 8; k++) prof[k] += tacc[k];
#undef SOLVE_MARK
}

// xl = Dinv (bl - Hpl^T xp)   (block_solver.hpp:461-481)
__global__ void __launch_bounds__(128) k_ba_backsub(BADev D) {
    const int l = (blockIdx.x * blockDim.x + threadIdx.x) / LM_LANES, sub = threadIdx.x % LM_LANES;
    const bool in = l < D.nMP, act = in && D.ptAct[l] && owned(D, l);
    double cl[3] = {0, 0, 0};
    const int eBeg = act ? D.lmStart[l] : 0, eEnd = act ? D.lmStart[l + 1] : 0;
    for (int a = eBeg + sub; a < eEnd; a += LM_LANES) {
        if (D.level[a] != 0) continue;
        const int p = D.poseIdx[D.eKF[a]];
        if (p < 0) continue;
        const double* B = D.Hpl + 18 * (size_t)a;
        const double* xq = D.xp + 6 * p;
#pragma unroll
        for (int j = 0; j < 3; j++) { double s = 0;
#pragma unroll
            for (int i = 0; i < 6; i++) s += B[3 * i + j] * xq[i]; cl[j] += s; }
    }
#pragma unroll
    for (int j = 0; j < 3; j++) { cl[j] += __shfl_xor_sync(0xffffffffu, cl[j], 1); cl[j] += __shfl_xor_sync(0xffffffffu, cl[j], 2); }
    if (!in || sub) return;
    if (!act) { D.xl[3 * l] = 0; D.xl[3 * l + 1] = 0; D.xl[3 * l + 2] = 0; return; }
#pragma unroll
    for (int j = 0; j < 3; j++) cl[j] = D.bl[3 * l + j] - cl[j];
    const double* Di = D.Dinv + DINV_LD * (size_t)l;
#pragma unroll
    for (int i = 0; i < 3; i++) D.xl[3 * l + i] = Di[3 * i] * cl[0] + Di[3 * i + 1] * cl[1] + Di[3 * i + 2] * cl[2];
}

__device__ __noinline__ Pose pose_oplus_ba(const Pose& est, const double* u) { return pose_oplus(est, u); }

// push() + oplus (base_vertex.h:96-99, types_six_dof_expmap.h:73-76, types_sba.h:52-56)
__global__ void __launch_bounds__(256) k_ba_update(BADev D) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < D.nKF) { const Pose T = D.pose[i]; D.poseBak[i] = T; const int p = D.poseIdx[i]; if (p >= 0) D.pose[i] = pose_oplus_ba(T, D.xp + 6 * p); }
    if (i < D.nMP) {
        const double x = D.X[3 * i], y = D.X[3 * i + 1], z = D.X[3 * i + 2];
        D.Xbak[3 * i] = x; D.Xbak[3 * i + 1] = y; D.Xbak[3 * i + 2] = z;
        if (D.ptAct[i] && owned(D, i)) { D.X[3 * i] = x + D.xl[3 * i]; D.X[3 * i + 1] = y + D.xl[3 * i + 1]; D.X[3 * i + 2] = z + D.xl[3 * i + 2]; }
    }
}
// pop()
__global__ void __launch_bounds__(256) k_ba_restore(BADev D) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < D.nKF) D.pose[i] = D.poseBak[i];
    if (i < D.nMP) { D.X[3 * i] = D.Xbak[3 * i]; D.X[3 * i + 1] = D.Xbak[3 * i + 1]; D.X[3 * i + 2] = D.Xbak[3 * i + 2]; }
}

// computeScale: sum_j x_j (lambda x_j + b_j); the pose part is added by rank 0 only (replicated), landmarks by their owner
__global__ void __launch_bounds__(256) k_ba_scale(BADev D, double* out) {
    __shared__ double sh[32];
    const double lambda = D.scal[4];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    double v = 0;
    if (i < D.n && D.rank == 0) v = D.xp[i] * (lambda * D.xp[i] + D.bpr[i]);
    const int j = i - D.n;
    if (j >= 0 && j < 3 * D.nMP) { const int l = j / 3; if (D.ptAct[l] && owned(D, l)) v = D.xl[j] * (lambda * D.xl[j] + D.bl[j]); }
    double tot;
    if (grid_sum(v, D.part, D.ticket, sh, &tot)) *out = tot;
}

// outlier test of src/Optimizer.cpp:384 / :411: chi2 of the LAST COMPUTED error (g2o keeps e->_error from the last
// computeActiveErrors, which may belong to a rejected trial) or non-positive depth in the rig frame
__global__ void __launch_bounds__(256) k_ba_classify(BADev D, uint8_t* flag) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= D.nE) return;
    double Xc[3];
    pose_map(D.pose[D.eKF[e]], D.X + 3 * D.eMP[e], Xc);
    const double chi = D.obs[3 * e + 2] * (D.err[2 * e] * D.err[2 * e] + D.err[2 * e + 1] * D.err[2 * e + 1]);
    flag[e] = (chi > 5.991 || !(Xc[2] > 0.0)) ? 1 : 0;
}

// ---------------------------------------------------------------------------------------------- one-shot NVLink all-reduce
// Multi-GPU LocalBA: every rank owns an exchange buffer [payload doubles | flags] that all peers map (CUDA IPC). After the Schur
// kernel has written the rank's partial [S | g | bpr | tail] into its own buffer, k_ba_xchg_signal publishes `epoch` in every peer's
// flag slot for this rank (system-scope release); k_ba_xchg_reduce waits until all peers have published `epoch`, then every rank sums
// the payloads of all ranks in rank order (identical result everywhere) into its private S / g / bpr / tail and adds lambda to the
// diagonal. One 0.7 MB exchange per LM trial instead of five NCCL calls; a bounded spin turns a lost peer into an error, not a hang.
struct XchgPeers { const double* payload[8]; volatile unsigned* flags[8]; int n, rank; };
__global__ void k_ba_xchg_signal(XchgPeers P, unsigned epoch) {
    if (threadIdx.x < P.n) {
        __threadfence_system();
        P.flags[threadIdx.x][P.rank] = epoch;   // slot `rank` of peer threadIdx.x's flag array
        __threadfence_system();
    }
}
__global__ void __launch_bounds__(256) k_ba_xchg_reduce(XchgPeers P, unsigned epoch, double* dst, size_t count, int n, const double* lambdaPtr, int* err) {
    __shared__ int ok;
    const double lambda = *lambdaPtr;
    if (threadIdx.x == 0) {
        ok = 1;
        volatile unsigned* mine = P.flags[P.rank];
        for (int r = 0; r < P.n; r++) {
            long long spins = 0;
            while ((int)(mine[r] - epoch) < 0) { if (++spins > (1ll << 26)) { ok = 0; break; } __nanosleep(64); }   // a fast peer may already be one epoch ahead
            if (!ok) break;
        }
        __threadfence_system();
    }
    __syncthreads();
    if (!ok) { if (threadIdx.x == 0) *err = 1; return; }
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) {
        double s = 0;
        for (int r = 0; r < P.n; r++) s += __ldcv(P.payload[r] + i);
        if (i < (size_t)n * n && (i / n) == (i % n)) s += lambda;
        dst[i] = s;
    }
}

// The scalars of a trial (chi2, scale; lambda_init's max diagonal) travel the same way: <= 4 doubles per rank in a double-buffered slot of
// the exchange region, one warp, one launch, fixed rank order (instead of a ~30 us ncclAllReduce per trial and per iteration).
struct SmallPeers { volatile unsigned* flags[8]; const double* slot[8]; double* mine; int n, rank; };
__global__ void k_ba_small_xchg(SmallPeers P, unsigned epoch, const double* src, double* dst, int count, int isMax, int* err) {
    const int t = threadIdx.x;
    double* slot = P.mine + (epoch & 1) * 4;
    if (t < count) slot[t] = src[t];
    __threadfence_system();
    __syncwarp();
    if (t < P.n) P.flags[t][P.rank] = epoch;
    __threadfence_system();
    bool ok = true;
    if (t < P.n) {
        volatile unsigned* mine = P.flags[P.rank];
        long long spins = 0;
        while ((int)(mine[t] - epoch) < 0) { if (++spins > (1ll << 26)) { ok = false; break; } __nanosleep(32); }
    }
    ok = __all_sync(0xffffffffu, ok);
    __threadfence_system();
    if (!ok) { if (t == 0) *err = 1; return; }
    if (t < count) {
        double v = __ldcv(P.slot[0] + (epoch & 1) * 4 + t);
        for (int r = 1; r < P.n; r++) { const double u = __ldcv(P.slot[r] + (epoch & 1) * 4 + t); v = isMax ? fmax(v, u) : v + u; }
        dst[t] = v;
    }
}
// multi-GPU: a rank classifies the edges of its own landmarks; the flags go to the caller's edge positions of a zeroed array that is max-reduced
__global__ void __launch_bounds__(256) k_ba_scatter_flags(int nLocal, const int* __restrict__ perm, const uint8_t* __restrict__ flag, uint8_t* __restrict__ out) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < nLocal) out[perm[s]] = flag[s];
}

}  // namespace cslam

// =================================================================================================== host side
using namespace cslam;

// ---- NCCL through dlopen (libnccl.so.2 is already mapped when torch.distributed is in use); no link-time dependency
typedef struct { char internal[128]; } nccl_uid_t;
struct NcclApi {
    void* h = nullptr;
    int (*GetUniqueId)(nccl_uid_t*) = nullptr;
    int (*CommInitRank)(nccl_comm_t*, int, nccl_uid_t, int) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*CommDestroy)(nccl_comm_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
static NcclApi* nccl_api() {
    static NcclApi api; static bool tried = false;
    if (tried) return api.h ? &api : nullptr;
    tried = true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) { api.h = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (api.h) break; }
    if (!api.h) return nullptr;
    api.GetUniqueId = (int (*)(nccl_uid_t*))dlsym(api.h, "ncclGetUniqueId");
    api.CommInitRank = (int (*)(nccl_comm_t*, int, nccl_uid_t, int))dlsym(api.h, "ncclCommInitRank");
    api.AllReduce = (int (*)(const void*, void*, size_t, int, int, nccl_comm_t, cudaStream_t))dlsym(api.h, "ncclAllReduce");
    api.AllGather = (int (*)(const void*, void*, size_t, int, nccl_comm_t, cudaStream_t))dlsym(api.h, "ncclAllGather");
    api.CommDestroy = (int (*)(nccl_comm_t))dlsym(api.h, "ncclCommDestroy");
    api.GetErrorString = (const char* (*)(int))dlsym(api.h, "ncclGetErrorString");
    if (!api.GetUniqueId || !api.CommInitRank || !api.AllReduce || !api.CommDestroy) { dlclose(api.h); api.h = nullptr; return nullptr; }
    return &api;
}
enum { NCCL_U8 = 1, NCCL_I32 = 2, NCCL_F64 = 8, NCCL_SUM = 0, NCCL_MAX = 2 };
enum { BK_ERRORS = 0, BK_LIN_POINTS, BK_LIN_POSES, BK_DINV, BK_SCHUR, BK_XCHG, BK_SOLVE, BK_BACKSUB, BK_UPDATE, BK_SCALE, BK_END, BK_COUNT };
static const char* kBaKindNames[BK_COUNT] = {"k_ba_errors", "k_ba_lin_points", "k_ba_lin_poses", "k_ba_dinv", "k_ba_schur", "exchange", "k_ba_solve", "k_ba_backsub", "k_ba_update", "k_ba_scale", "end"};

// Dynamic shared memory of k_ba_solve: [staged panels 2 x NB x ldp] + y[n]. y alone caps the system at n = SOLVE_DSMEM / 8 = 26112 (4352 free key frames).
static const int SOLVE_DSMEM = 204 * 1024;
static const size_t SOLVE_STAGE_BYTES = 200 * 1024;   // the panels are staged when they and y fit in this

// Shared-memory plan of k_ba_solve for an n x n system with panel stride ldp. stage: -1 = stage when it fits, 0 = panels read from L2, 1 = staged.
static int solve_plan(int n, int ldp, int stage, int* stageOut, size_t* dsmem) {
    const size_t panel = 2 * (size_t)LD_NB * ldp * 8, ybytes = (size_t)n * 8;
    if (ybytes > (size_t)SOLVE_DSMEM) { set_error("reduced camera system n = %d exceeds the solver's shared-memory capacity (n <= %d, i.e. %d free key frames)", n, SOLVE_DSMEM / 8, SOLVE_DSMEM / 48); return CSLAM_E_CAPACITY; }
    const bool fits = panel + ybytes <= SOLVE_STAGE_BYTES;
    if (stage == 1 && !fits) { set_error("solve: staged panels do not fit in shared memory at n = %d", n); return CSLAM_E_BADARG; }
    *stageOut = stage < 0 ? (fits ? 1 : 0) : stage;
    *dsmem = (*stageOut ? panel : 0) + ybytes;
    return 0;
}

static cudaLaunchConfig_t solve_config(cudaLaunchAttribute* at, int cluster, size_t dsmem, cudaStream_t s) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(cluster); cfg.blockDim = dim3(SOLVE_T); cfg.dynamicSmemBytes = dsmem; cfg.stream = s;
    at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = cluster; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cfg;
}

// The one launch of k_ba_solve (LM trials and cslam_ba_solve_dense): one cluster of `cluster` CTAs factors R.S / R.g in place, writes R.xp and
// sets R.scal[3] = 1 on a zero / non-finite pivot.
static int launch_solve(cslam_optimizer* o, const BADev& R, double* Lt, double* LDt, double* Minv, int ldp, int stage, int cluster, long long* prof) {
    int stg = 0; size_t dsmem = 0;
    if (int rc = solve_plan(R.n, ldp, stage, &stg, &dsmem)) return rc;
    cudaLaunchAttribute at[1];
    const cudaLaunchConfig_t cfg = solve_config(at, cluster, dsmem, o->stream);
    CSLAM_CUDA(cudaLaunchKernelEx(&cfg, k_ba_solve, R, Lt, LDt, Minv, ldp, stg, prof)); o->launches++;
    return 0;
}


extern "C" int cslam_optimizer_create(cslam_optimizer** out, int device) {
    if (!out) return CSLAM_E_BADARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { set_error("no CUDA device (this library has no CPU fallback)"); return CSLAM_E_NODEVICE; }
    if (device < 0 || device >= ndev) { set_error("device %d out of range", device); return CSLAM_E_BADARG; }
    CSLAM_CUDA(cudaSetDevice(device));
    cslam_optimizer* o = new cslam_optimizer; o->device = device;
    if (cudaStreamCreateWithFlags(&o->stream, cudaStreamNonBlocking) != cudaSuccess || cudaMallocHost(&o->h_scal, 16 * sizeof(double)) != cudaSuccess) {
        set_error("optimizer: stream / pinned allocation failed"); delete o; return CSLAM_E_CUDA;
    }
    if (const char* e = getenv("CSLAM_SOLVE_CLUSTER")) o->clusterSize = std::max(1, std::min(atoi(e), 16));
    if (o->clusterSize > 8) cudaFuncSetAttribute(k_ba_solve, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    cudaFuncSetAttribute(k_ba_solve, cudaFuncAttributeMaxDynamicSharedMemorySize, SOLVE_DSMEM);
    if (const char* e = getenv("CSLAM_BA_GRAPH")) o->useGraphs = atoi(e) != 0;
    *out = o;
    return CSLAM_OK;
}
static void release_pool(cslam_optimizer* o) { for (auto& c : o->chunks) cudaFree(c.p); o->chunks.clear(); }
extern "C" void cslam_optimizer_destroy(cslam_optimizer* o) {
    if (!o) return;
    cudaSetDevice(o->device);
    if (o->stream) cudaStreamSynchronize(o->stream);
    for (auto& p : o->peers) { if (p.base && !p.mine) cudaIpcCloseMemHandle(p.base); else if (p.base) cudaFree(p.base); }
    release_pool(o);
    if (o->comm && nccl_api()) nccl_api()->CommDestroy(o->comm);
    if (o->stream) cudaStreamDestroy(o->stream);
    if (o->h_scal) cudaFreeHost(o->h_scal);
    delete o;
}
extern "C" int64_t cslam_optimizer_launches(const cslam_optimizer* o) { return o ? o->launches : 0; }
extern "C" int cslam_optimizer_set_timing(cslam_optimizer* o, int enable) {
    if (!o) return CSLAM_E_BADARG;
    CSLAM_CUDA(cudaSetDevice(o->device));
    if (enable && o->ev.empty()) { o->ev.resize(64); o->evKind.resize(64); for (auto& e : o->ev) CSLAM_CUDA(cudaEventCreate(&e)); }
    o->timing = enable != 0; o->evUsed = 0;
    for (int i = 0; i < 16; i++) { o->kindMs[i] = 0; o->kindCount[i] = 0; }
    return CSLAM_OK;
}
extern "C" int cslam_optimizer_get_timing(const cslam_optimizer* o, int kind, const char** name, double* ms, int64_t* count) {
    if (!o || kind < 0 || kind >= BK_END) return CSLAM_E_BADARG;
    *name = kBaKindNames[kind]; *ms = o->kindMs[kind]; *count = o->kindCount[kind];
    return CSLAM_OK;
}

extern "C" int cslam_ba_solve_dense(cslam_optimizer* o, int n, const double* Sg, int stage, int cluster, double* x, int32_t* failed) {
    if (!o || !Sg || !x || !failed || n < 1 || stage < -1 || stage > 1 || cluster < 0 || cluster > 16) { set_error("cslam_ba_solve_dense: bad argument"); return CSLAM_E_BADARG; }
    const int C = cluster ? cluster : o->clusterSize;
    const int ldp = ((n + 1 + 8) + 3) & ~3;   // as cslam_local_ba sizes it
    int rc, stg = 0; size_t dsmem = 0;
    if ((rc = solve_plan(n, ldp, stage, &stg, &dsmem))) return rc;   // before anything touches Sg
    CSLAM_CUDA(cudaSetDevice(o->device));
    if (C > 8) CSLAM_CUDA(cudaFuncSetAttribute(k_ba_solve, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    {
        cudaLaunchAttribute at[1];
        const cudaLaunchConfig_t cfg = solve_config(at, C, dsmem, o->stream);
        int nc = 0;
        const cudaError_t e = cudaOccupancyMaxActiveClusters(&nc, k_ba_solve, &cfg);
        if (e != cudaSuccess || nc == 0) {
            cudaGetLastError();
            set_error("solve: a cluster of %d CTAs with %zu B of dynamic shared memory each cannot be scheduled on this device (%s)", C, dsmem, cudaGetErrorString(e));
            return CSLAM_E_BADARG;
        }
    }
    free_pool(o);
    BADev R; std::memset(&R, 0, sizeof(R));
    R.n = n;
    double *Lt = nullptr, *LDt = nullptr, *Minv = nullptr;
    if ((rc = dalloc(o, &R.S, (size_t)(n + 1) * n)) || (rc = dalloc(o, &R.xp, n)) || (rc = dalloc(o, &R.scal, 8, true)) || (rc = dalloc(o, &Lt, (size_t)LD_NB * ldp)) ||
        (rc = dalloc(o, &LDt, (size_t)LD_NB * ldp)) || (rc = dalloc(o, &Minv, (size_t)(n / LD_NB + 1) * LD_NB * LD_NB))) return rc;
    R.g = R.S + (size_t)n * n;
    CSLAM_CUDA(cudaMemcpyAsync(R.S, Sg, (size_t)(n + 1) * n * sizeof(double), cudaMemcpyHostToDevice, o->stream));
    if ((rc = launch_solve(o, R, Lt, LDt, Minv, ldp, stg, C, nullptr))) return rc;
    CSLAM_CUDA(cudaMemcpyAsync(x, R.xp, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, o->stream));
    CSLAM_CUDA(cudaMemcpyAsync(o->h_scal, R.scal + 3, sizeof(double), cudaMemcpyDeviceToHost, o->stream));
    CSLAM_CUDA(cudaStreamSynchronize(o->stream));
    *failed = o->h_scal[0] != 0.0;
    free_pool(o);
    return CSLAM_OK;
}

extern "C" int cslam_nccl_unique_id(uint8_t id128[128]) {
    NcclApi* a = nccl_api();
    if (!a) { set_error("libnccl.so.2 not found"); return CSLAM_E_NCCL; }
    nccl_uid_t id; int rc = a->GetUniqueId(&id);
    if (rc) { set_error("ncclGetUniqueId failed (%d)", rc); return CSLAM_E_NCCL; }
    std::memcpy(id128, id.internal, 128);
    return CSLAM_OK;
}

// Exchange buffers of the one-shot all-reduce: allocate, publish the CUDA IPC handle through ncclAllGather, map every peer.
static const size_t XCHG_FLAG_BYTES = 256;
static int setup_xchg(cslam_optimizer* o, size_t payloadBytes) {
    NcclApi* a = nccl_api();
    if (o->nranks > 8 || !a->AllGather) return 1;   // fall back to NCCL
    for (auto& p : o->peers) { if (p.base && !p.mine) cudaIpcCloseMemHandle(p.base); else if (p.base) cudaFree(p.base); }
    o->peers.assign(o->nranks, cslam_optimizer::Peer());
    void* mine = nullptr;
    const size_t bytes = 2 * ((payloadBytes + 255) & ~(size_t)255) + XCHG_FLAG_BYTES;   // two payload buffers (epoch parity) + the flag slots
    CSLAM_CUDA(cudaMalloc(&mine, bytes));
    CSLAM_CUDA(cudaMemset(mine, 0, bytes));
    cudaIpcMemHandle_t h;
    CSLAM_CUDA(cudaIpcGetMemHandle(&h, mine));
    cudaIpcMemHandle_t* dAll = nullptr;
    CSLAM_CUDA(cudaMalloc((void**)&dAll, sizeof(h) * o->nranks));
    CSLAM_CUDA(cudaMemcpy(dAll + o->rank, &h, sizeof(h), cudaMemcpyHostToDevice));
    int rc = a->AllGather(dAll + o->rank, dAll, sizeof(h), NCCL_U8, o->comm, o->stream);
    if (rc) { set_error("ncclAllGather (IPC handles) failed (%d)", rc); return CSLAM_E_NCCL; }
    std::vector<cudaIpcMemHandle_t> all(o->nranks);
    CSLAM_CUDA(cudaMemcpyAsync(all.data(), dAll, sizeof(h) * o->nranks, cudaMemcpyDeviceToHost, o->stream));
    CSLAM_CUDA(cudaStreamSynchronize(o->stream));
    cudaFree(dAll);
    bool ok = true;
    for (int r = 0; r < o->nranks; r++) {
        if (r == o->rank) { o->peers[r].base = mine; o->peers[r].mine = true; continue; }
        void* p = nullptr;
        if (cudaIpcOpenMemHandle(&p, all[r], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); ok = false; break; }
        o->peers[r].base = p;
    }
    // all ranks must agree on the path
    double* flag = nullptr;
    CSLAM_CUDA(cudaMalloc((void**)&flag, 8));
    const double v = ok ? 0.0 : 1.0;
    CSLAM_CUDA(cudaMemcpy(flag, &v, 8, cudaMemcpyHostToDevice));
    rc = a->AllReduce(flag, flag, 1, NCCL_F64, NCCL_SUM, o->comm, o->stream);
    double bad = 1;
    CSLAM_CUDA(cudaMemcpyAsync(&bad, flag, 8, cudaMemcpyDeviceToHost, o->stream));
    CSLAM_CUDA(cudaStreamSynchronize(o->stream));
    cudaFree(flag);
    if (rc || bad != 0.0) return 1;
    o->xchgBytes = payloadBytes; o->oneShot = true; o->epoch = 0; o->epoch2 = 0;
    return 0;
}

extern "C" int cslam_optimizer_init_nccl(cslam_optimizer* o, const uint8_t id128[128], int rank, int nranks) {
    if (!o || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return CSLAM_E_BADARG;
    NcclApi* a = nccl_api();
    if (!a) { set_error("libnccl.so.2 not found"); return CSLAM_E_NCCL; }
    CSLAM_CUDA(cudaSetDevice(o->device));
    nccl_uid_t id; std::memcpy(id.internal, id128, 128);
    int rc = a->CommInitRank(&o->comm, nranks, id, rank);
    if (rc) { set_error("ncclCommInitRank failed: %s", a->GetErrorString ? a->GetErrorString(rc) : "?"); return CSLAM_E_NCCL; }
    o->rank = rank; o->nranks = nranks;
    return CSLAM_OK;
}

// Per-edge input conversion on the device (was a host loop): cube face of the key point (CamModelGeneral::FaceInCubemap(cv::Point2f),
// float arithmetic as the reference), position inside the face as double (GetPosInFace<double>), information weight; s = position in the
// landmark-sorted order, perm[s] = the caller's edge index (perm == nullptr: the caller's order is already grouped by landmark).
__global__ void __launch_bounds__(256) k_ba_prep_edges(int nE, const int* __restrict__ perm, const float2* __restrict__ kp, const float* __restrict__ isig, int faceW, int faceH,
                                                       double* __restrict__ obs, int8_t* __restrict__ face, int* __restrict__ bad) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nE) return;
    const int e = perm ? perm[s] : s;
    const float2 k = kp[e];
    const float fi = __fdiv_rn(k.x, (float)faceW), fj = __fdiv_rn(k.y, (float)faceH);
    int f = -1;
    if (fi >= 0 && fi < 1 && fj >= 1 && fj < 2) f = 1;
    else if (fi >= 1 && fi < 2 && fj >= 0 && fj < 1) f = 3;
    else if (fi >= 1 && fi < 2 && fj >= 1 && fj < 2) f = 0;
    else if (fi >= 1 && fi < 2 && fj >= 2 && fj < 3) f = 4;
    else if (fi >= 2 && fi < 3 && fj >= 1 && fj < 2) f = 2;
    if (f < 0) atomicMin(bad, e);
    face[s] = (int8_t)f;
    obs[3 * s] = (double)k.x - floor((double)k.x / faceW) * faceW;
    obs[3 * s + 1] = (double)k.y - floor((double)k.y / faceH) * faceH;
    obs[3 * s + 2] = (double)isig[e];
}
__global__ void __launch_bounds__(256) k_ba_prep_points(int n3, const float* __restrict__ in, double* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n3) out[i] = (double)in[i];
}

namespace {
struct BAHost {
    cslam_optimizer* o; BADev D; cslam_ba_result* res;
    const int* perm = nullptr;        // sorted edge position -> caller's edge index; nullptr = identity (input already grouped by landmark)
    std::vector<uint8_t> level; std::vector<int> poseIdx; std::vector<uint8_t> ptAct, fixed;
    int* d_poseIdx = nullptr; uint8_t* d_ptAct = nullptr; uint8_t* d_flag = nullptr; int* d_pact = nullptr;
    double* Lt = nullptr; double* LDt = nullptr; double* Minv = nullptr; int ldp = 0;   // panel buffers, inverses of the diagonal blocks' unit factors
    double* red = nullptr;            // private reduce buffer [S | g | bpr | tail]
    double* HppFull = nullptr;        // multi-GPU: all-reduced copy of the pose blocks for computeLambdaInit
    size_t xstride = 0;               // one-shot path: doubles between the two payload buffers of an exchange region
    int* d_xerr = nullptr;
    long long* d_prof = nullptr;      // CSLAM_BA_PROFILE=1: clock64 per solver phase (debug)
    double lambda = -1, ni = 2; int nBad = 0; int iterations = 0, trials = 0;
    bool errorsCurrent = false; double lastChi = 0;   // D.err / chi2 belong to the current state (set by an accepted trial)
    const volatile uint8_t* stop = nullptr;
    const int* h_eMP = nullptr; const int* h_eKF = nullptr; int nActive = 0;   // landmark-sorted edge endpoints on the host
    bool useOneShot = false;
    bool terminate() const { return stop ? (*stop != 0) : false; }
    int grid(int n, int t = 256) const { return std::max(1, cdiv(n, t)); }
    size_t payload() const { return (size_t)D.n * D.n + 2 * (size_t)D.n + 4; }

    int allreduce(double* buf, size_t count, int op) {
        if (o->nranks <= 1) return 0;
        int rc = nccl_api()->AllReduce(buf, buf, count, NCCL_F64, op, o->comm, o->stream);
        if (rc) { set_error("ncclAllReduce failed (%d)", rc); return CSLAM_E_NCCL; }
        return 0;
    }
    // <= 4 doubles, in place: the one-shot path when the peer views exist, NCCL otherwise
    int allreduce_small(double* buf, int count, bool isMax) {
        if (o->nranks <= 1) return 0;
        if (!useOneShot) return allreduce(buf, count, isMax ? NCCL_MAX : NCCL_SUM);
        SmallPeers P; P.n = o->nranks; P.rank = o->rank;
        const size_t off = 2 * xstride * 8;
        for (int r = 0; r < o->nranks; r++) { P.flags[r] = (volatile unsigned*)((char*)o->peers[r].base + off + 64); P.slot[r] = (const double*)((char*)o->peers[r].base + off + 128); }
        P.mine = (double*)((char*)o->peers[o->rank].base + off + 128);
        k_ba_small_xchg<<<1, 32, 0, o->stream>>>(P, ++o->epoch2, buf, buf, count, isMax ? 1 : 0, d_xerr); o->launches++;
        return 0;
    }
    int fetch(const double* src, int count) {
        CSLAM_CUDA(cudaMemcpyAsync(o->h_scal, src, count * sizeof(double), cudaMemcpyDeviceToHost, o->stream));
        CSLAM_CUDA(cudaStreamSynchronize(o->stream));
        return 0;
    }
    void bind(unsigned epoch = 0) {   // partial system of this rank goes to `w` (exchange payload of this epoch on the one-shot path), the reduced one lives in `red`
        double* w = (o->nranks > 1 && useOneShot) ? (double*)o->peers[o->rank].base + (epoch & 1) * xstride : red;
        D.S = w; D.g = w + (size_t)D.n * D.n; D.bpr = D.g + D.n; D.tail = D.bpr + D.n;
    }
    BADev reducedView() const { BADev R = D; R.S = red; R.g = red + (size_t)D.n * D.n; R.bpr = R.g + D.n; R.tail = R.bpr + D.n; return R; }

    // initializeOptimization(level 0): active edges, active vertices, compact pose indices (sparse_optimizer.cpp:206-267,166-190)
    int initialize() {
        std::vector<int> pAct(D.nKF + 1, 0);   // [nKF] = this rank has an active edge
        std::fill(ptAct.begin(), ptAct.end(), 0);
        const int* eMP = h_eMP; const int* eKF = h_eKF;
        nActive = 0;
        for (int e = 0; e < D.nE; e++) if (level[e] == 0) { pAct[eKF[e]] = 1; ptAct[eMP[e]] = 1; nActive++; }
        pAct[D.nKF] = nActive > 0;
        if (o->nranks > 1) {   // a rank sees the edges of its own landmarks only: pose activity and "anything to optimize" are global facts
            CSLAM_CUDA(cudaMemcpyAsync(d_pact, pAct.data(), (D.nKF + 1) * sizeof(int), cudaMemcpyHostToDevice, o->stream));
            int rc = nccl_api()->AllReduce(d_pact, d_pact, D.nKF + 1, NCCL_I32, NCCL_MAX, o->comm, o->stream);
            if (rc) { set_error("ncclAllReduce (pose activity) failed (%d)", rc); return CSLAM_E_NCCL; }
            CSLAM_CUDA(cudaMemcpyAsync(pAct.data(), d_pact, (D.nKF + 1) * sizeof(int), cudaMemcpyDeviceToHost, o->stream));
            CSLAM_CUDA(cudaStreamSynchronize(o->stream));
            nActive = pAct[D.nKF];   // only tested against zero
        }
        int nP = 0;
        for (int k = 0; k < D.nKF; k++) poseIdx[k] = (pAct[k] && !fixed[k]) ? nP++ : -1;
        D.nP = nP; D.n = 6 * nP;
        CSLAM_CUDA(cudaMemcpyAsync(d_poseIdx, poseIdx.data(), D.nKF * sizeof(int), cudaMemcpyHostToDevice, o->stream));
        CSLAM_CUDA(cudaMemcpyAsync(d_ptAct, ptAct.data(), D.nMP, cudaMemcpyHostToDevice, o->stream));
        CSLAM_CUDA(cudaMemcpyAsync(D.level, level.data(), D.nE, cudaMemcpyHostToDevice, o->stream));
        errorsCurrent = false;   // level / robust kernel changed
        bind();
        drop_graph();   // the captured trial bakes in nP / n / the level array's meaning
        return 0;
    }
    int errors_chi2(double* chi) {   // computeActiveErrors + activeRobustChi2
        k_ba_errors<<<grid(D.nE), 256, 0, o->stream>>>(D, D.scal); o->launches++;
        int rc;
        if ((rc = allreduce_small(D.scal, 1, false))) return rc;
        if ((rc = fetch(D.scal, 1))) return rc;
        *chi = o->h_scal[0];
        return 0;
    }
    int build_system() {
        k_ba_lin_points<<<grid(D.nMP * LM_LANES, 128), 128, 0, o->stream>>>(D); o->launches++;
        tick(BK_LIN_POSES);
        if (D.nQ > 0) { k_ba_lin_poses<<<dim3(D.nQ, POSE_SPLIT), 256, 0, o->stream>>>(D); o->launches++; }
        CSLAM_CUDA(cudaGetLastError());
        return 0;
    }
    int lambda_init(double* lam) {
        int rc;
        CSLAM_CUDA(cudaMemsetAsync(D.scal + 2, 0, sizeof(double), o->stream));
        BADev M = D;
        if (o->nranks > 1 && D.nP > 0) {   // computeLambdaInit needs the full pose blocks: sum a COPY of the partial blocks once per optimize()
            CSLAM_CUDA(cudaMemcpyAsync(HppFull, D.Hpp, (size_t)D.nP * 36 * 8, cudaMemcpyDeviceToDevice, o->stream));
            if ((rc = allreduce(HppFull, (size_t)D.nP * 36, NCCL_SUM))) return rc;
            M.Hpp = HppFull;
        }
        k_ba_maxdiag<<<grid(D.nP * 6 + D.nMP * 3), 256, 0, o->stream>>>(M); o->launches++;
        if ((rc = allreduce_small(D.scal + 2, 1, true))) return rc;
        if ((rc = fetch(D.scal, 4))) return rc;
        *lam = 1e-5 * o->h_scal[2];
        return 0;
    }
    // ---- optional per-kernel timing (cslam_optimizer_set_timing): CUDA events between launches, accumulated per kernel kind
    void tick(int kind) {
        if (!o->timing || o->evUsed >= (int)o->ev.size()) return;
        cudaEventRecord(o->ev[o->evUsed], o->stream); o->evKind[o->evUsed++] = kind;
    }
    void collect() {
        for (int i = 0; i + 1 < o->evUsed; i++) {
            float ms = 0;
            if (o->evKind[i] != BK_END && cudaEventElapsedTime(&ms, o->ev[i], o->ev[i + 1]) == cudaSuccess) { o->kindMs[o->evKind[i]] += ms; o->kindCount[o->evKind[i]]++; }
        }
        o->evUsed = 0;
    }
    // One LM trial on the stream: lambda -> device, BlockSolver::solve (Dinv, Schur, [exchange], reduced solve, back substitution), push + oplus,
    // computeActiveErrors + activeRobustChi2, computeScale, the four scalars -> pinned host memory. Single-GPU trials are replayed as ONE CUDA graph.
    int enqueue_trial() {
        int rc;
        CSLAM_CUDA(cudaMemcpyAsync(D.scal + 4, o->h_scal + 8, sizeof(double), cudaMemcpyHostToDevice, o->stream));   // h_scal[8] = lambda
        tick(BK_DINV);
        k_ba_dinv<<<grid(D.nMP), 256, 0, o->stream>>>(D); o->launches++;
        BADev SV = D;
        if (D.n > 0) {
            const bool multi = o->nranks > 1;
            const unsigned ep = (multi && useOneShot) ? ++o->epoch : 0;
            bind(ep);
            tick(BK_SCHUR);
            k_ba_schur<<<dim3(D.nQ, D.nQ), SCHUR_T, 0, o->stream>>>(D, multi ? 0 : 1); o->launches++;
            BADev R = D;
            if (multi) {
                R = reducedView();
                tick(BK_XCHG);
                if (useOneShot) {
                    XchgPeers P; P.n = o->nranks; P.rank = o->rank;
                    const size_t off = 2 * xstride * 8;
                    for (int r = 0; r < o->nranks; r++) { P.payload[r] = (const double*)o->peers[r].base + (ep & 1) * xstride; P.flags[r] = (volatile unsigned*)((char*)o->peers[r].base + off); }
                    k_ba_xchg_signal<<<1, 32, 0, o->stream>>>(P, ep); o->launches++;
                    k_ba_xchg_reduce<<<std::min(148, grid((int)std::min<size_t>(payload(), 1u << 30))), 256, 0, o->stream>>>(P, ep, red, payload(), D.n, D.scal + 4, d_xerr); o->launches++;
                } else {
                    CSLAM_CUDA(cudaMemcpyAsync(red, D.S, payload() * 8, cudaMemcpyDeviceToDevice, o->stream));
                    if ((rc = allreduce(red, payload(), NCCL_SUM))) return rc;
                    k_ba_add_lambda_launch(R);
                }
                SV.bpr = R.bpr;
            }
            CSLAM_CUDA(cudaMemsetAsync(D.scal + 3, 0, sizeof(double), o->stream));
            tick(BK_SOLVE);
            if ((rc = launch_solve(o, R, Lt, LDt, Minv, ldp, -1, o->clusterSize, d_prof))) return rc;
        }
        tick(BK_BACKSUB);
        k_ba_backsub<<<grid(D.nMP * LM_LANES, 128), 128, 0, o->stream>>>(D); o->launches++;
        tick(BK_UPDATE);
        k_ba_update<<<grid(std::max(D.nKF, D.nMP)), 256, 0, o->stream>>>(D); o->launches++;
        tick(BK_ERRORS);
        k_ba_errors<<<grid(D.nE), 256, 0, o->stream>>>(D, D.scal); o->launches++;
        tick(BK_SCALE);
        k_ba_scale<<<grid(D.n + 3 * D.nMP), 256, 0, o->stream>>>(SV, D.scal + 1); o->launches++;
        tick(BK_END);
        if ((rc = allreduce_small(D.scal, 2, false))) return rc;
        CSLAM_CUDA(cudaMemcpyAsync(o->h_scal, D.scal, 4 * sizeof(double), cudaMemcpyDeviceToHost, o->stream));
        CSLAM_CUDA(cudaGetLastError());
        return 0;
    }
    cudaGraphExec_t trialGraph = nullptr;
    void drop_graph() { if (trialGraph) { cudaGraphExecDestroy(trialGraph); trialGraph = nullptr; } }
    int run_trial() {
        int rc;
        o->h_scal[8] = lambda;
        const bool useGraph = o->nranks == 1 && !o->timing && o->useGraphs;
        if (useGraph) {
            if (!trialGraph) {
                cudaGraph_t g = nullptr;
                const int64_t l0 = o->launches;
                CSLAM_CUDA(cudaStreamBeginCapture(o->stream, cudaStreamCaptureModeThreadLocal));
                rc = enqueue_trial();
                cudaError_t ce = cudaStreamEndCapture(o->stream, &g);
                if (rc) { if (g) cudaGraphDestroy(g); return rc; }
                CSLAM_CUDA(ce);
                CSLAM_CUDA(cudaGraphInstantiate(&trialGraph, g, 0));
                cudaGraphDestroy(g);
                launchesPerTrial = o->launches - l0; o->launches = l0;
            }
            CSLAM_CUDA(cudaGraphLaunch(trialGraph, o->stream));
            o->launches += launchesPerTrial;
        } else if ((rc = enqueue_trial())) return rc;
        CSLAM_CUDA(cudaStreamSynchronize(o->stream));
        if (o->timing) collect();
        return 0;
    }
    int64_t launchesPerTrial = 0;
    void k_ba_add_lambda_launch(const BADev& R);
    // OptimizationAlgorithmLevenberg::solve ; result 0 OK, 1 Terminate
    int lm_iteration(int iteration, int* result) {
        int rc; double currentChi = 0;
        tick(BK_ERRORS);
        // computeActiveErrors + activeRobustChi2: after an accepted trial the errors and chi2 of this very state are already on the device
        // (the trial evaluated them; same kernel, same inputs -> same bits), so only the first iteration and the ones after a rejection compute
        if (errorsCurrent) currentChi = lastChi;
        else if ((rc = errors_chi2(&currentChi))) return rc;
        const double iniChi = currentChi; double tempChi = currentChi;
        tick(BK_LIN_POINTS);
        if ((rc = build_system())) return rc;
        tick(BK_END);
        if (iteration == 0) { if ((rc = lambda_init(&lambda))) return rc; ni = 2; nBad = 0; }
        double rho = 0; int qmax = 0; int accepted = 0;
        do {
            if ((rc = run_trial())) return rc;
            tempChi = o->h_scal[0];
            bool ok2 = o->h_scal[3] == 0.0;
            trials++;
            if (!ok2) tempChi = DBL_MAX;
            rho = currentChi - tempChi;
            const double scale = o->h_scal[1] + 1e-3;
            rho /= scale;
            if (rho > 0 && std::isfinite(tempChi) && ok2) {
                double alpha = 1. - std::pow((2 * rho - 1), 3);
                alpha = std::min(alpha, 2. / 3.);
                lambda *= std::max(1. / 3., alpha); ni = 2; currentChi = tempChi; accepted = 1;
                errorsCurrent = true; lastChi = tempChi;
            } else {
                errorsCurrent = false;   // pop(): the state is the old one again, the error array holds the trial's
                lambda *= ni; ni *= 2;
                k_ba_restore<<<grid(std::max(D.nKF, D.nMP)), 256, 0, o->stream>>>(D); o->launches++;
                if (!ok2) rho = -1;
            }
            qmax++;
        } while (rho < 0 && qmax < 10 && !terminate());
        if (res && res->lm_log && iterations < res->log_cap) {
            double* L = res->lm_log + 4 * iterations; L[0] = currentChi; L[1] = lambda; L[2] = qmax; L[3] = accepted;
        }
        iterations++;
        *result = 0;
        if (qmax == 10 || rho == 0) { *result = 1; return 0; }
        if ((iniChi - currentChi) * 1e3 < iniChi) nBad++; else nBad = 0;
        if (nBad >= 3) *result = 1;
        return 0;
    }
    int optimize(int its) {
        if (nActive == 0) return 0;   // g2o: "0 vertices to optimize"
        int result = 0;
        for (int i = 0; i < its && !terminate() && result == 0; i++) { int rc = lm_iteration(i, &result); if (rc) return rc; }
        if (o->nranks > 1 && useOneShot) {
            int xe = 0;
            CSLAM_CUDA(cudaMemcpyAsync(&xe, d_xerr, sizeof(int), cudaMemcpyDeviceToHost, o->stream));
            CSLAM_CUDA(cudaStreamSynchronize(o->stream));
            if (xe) { set_error("one-shot all-reduce: a peer never signalled (timeout)"); return CSLAM_E_NCCL; }
        }
        return 0;
    }
    int classify(std::vector<uint8_t>& flags) {   // flags of this rank's edges (all edges on one GPU)
        k_ba_classify<<<grid(D.nE), 256, 0, o->stream>>>(D, d_flag); o->launches++;
        flags.resize(D.nE);
        CSLAM_CUDA(cudaMemcpyAsync(flags.data(), d_flag, D.nE, cudaMemcpyDeviceToHost, o->stream));
        CSLAM_CUDA(cudaStreamSynchronize(o->stream));
        return 0;
    }
};
__global__ void __launch_bounds__(256) k_ba_add_lambda(double* S, int n, double lambda) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) S[(size_t)i * n + i] += lambda;
}
void BAHost::k_ba_add_lambda_launch(const BADev& R) { k_ba_add_lambda<<<grid(R.n), 256, 0, o->stream>>>(R.S, R.n, lambda); o->launches++; }

// non-owner points are stale on a rank: every point is taken from its owner (sum of owner ? X : 0)
__global__ void __launch_bounds__(256) k_ba_mask_points(BADev D) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l < D.nMP && !owned(D, l)) { D.X[3 * l] = 0; D.X[3 * l + 1] = 0; D.X[3 * l + 2] = 0; }
}
}  // namespace

extern "C" int cslam_local_ba(cslam_optimizer* o, cslam_ba_problem* p, const volatile uint8_t* stop_flag, int its1, int its2, cslam_ba_result* r) {
    if (!o || !p || p->n_kf <= 0 || p->n_mp < 0 || p->n_edges < 0 || !p->Tcw || !p->kf_fixed || (p->n_mp && !p->points)) { set_error("cslam_local_ba: bad problem"); return CSLAM_E_BADARG; }
    if (p->face_w != p->face_h || p->face_w <= 0) { set_error("cube faces must be square"); return CSLAM_E_BADARG; }
    CSLAM_CUDA(cudaSetDevice(o->device));
    free_pool(o);
    const bool hostProf = getenv("CSLAM_BA_PROFILE") != nullptr;
    auto tNow = []() { return std::chrono::steady_clock::now(); };
    auto tMs = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
    const auto tp0 = tNow();
    const int nKF = p->n_kf, nMP = p->n_mp, nEg = p->n_edges;   // nEg: the caller's edges; nE below: the edges this rank works on
    if (r) { r->iterations = 0; r->trials = 0; if (r->outlier) std::memset(r->outlier, 0, nEg); }
    if (stop_flag && *stop_flag) return CSLAM_OK;   // src/Optimizer.cpp:359-361
    BAHost H; H.o = o; H.res = r; H.stop = stop_flag;
    BADev& D = H.D; std::memset(&D, 0, sizeof(D));
    D.nKF = nKF; D.nMP = nMP; D.f = p->face_w / 2.0; D.rank = o->rank; D.nranks = o->nranks;
    const float dlt = (float)std::sqrt(5.991); D.delta = (double)dlt; D.dsqr = D.delta * D.delta; D.robust = 1;
    // ---- edges sorted by landmark (stable), CSR by landmark and by keyframe. Host work is two passes over the endpoint arrays (in scratch
    // vectors that live in the optimizer object: no page faults per call); the per-edge float work happens on the device (k_ba_prep_edges).
    cslam_optimizer::HostScratch& hs = o->hs;
    hs.lmStart.assign(nMP + 1, 0);
    // Multi-GPU: landmark l (with all its edges) belongs to rank l % nranks; a rank works on the edges of its own landmarks ONLY, so every
    // per-edge kernel, the co-observation lists and the Schur work shrink by 1 / nranks; the reduced camera system is what gets exchanged.
    const bool multi = o->nranks > 1;
    bool grouped = !multi;
    int nLocal = 0;
    for (int e = 0; e < nEg; e++) {
        const int l = p->edge_mp[e], k = p->edge_kf[e];
        if (l < 0 || l >= nMP || k < 0 || k >= nKF) { set_error("edge %d references a vertex out of range", e); return CSLAM_E_BADARG; }
        if (multi && (l % o->nranks) != o->rank) continue;
        hs.lmStart[l + 1]++; nLocal++;
        if (e && l < p->edge_mp[e - 1]) grouped = false;
    }
    const int nE = nLocal;
    D.nE = nE;
    for (int l = 0; l < nMP; l++) hs.lmStart[l + 1] += hs.lmStart[l];
    if (grouped) { H.perm = nullptr; H.h_eMP = p->edge_mp; H.h_eKF = p->edge_kf; }
    else {
        hs.perm.resize(nE); hs.eMP.resize(nE); hs.eKF.resize(nE); hs.fill.assign(hs.lmStart.begin(), hs.lmStart.end() - 1);
        for (int e = 0; e < nEg; e++) { const int l = p->edge_mp[e]; if (!multi || (l % o->nranks) == o->rank) hs.perm[hs.fill[l]++] = e; }
        for (int s = 0; s < nE; s++) { const int e = hs.perm[s]; hs.eMP[s] = p->edge_mp[e]; hs.eKF[s] = p->edge_kf[e]; }
        H.perm = hs.perm.data(); H.h_eMP = hs.eMP.data(); H.h_eKF = hs.eKF.data();
    }
    hs.peStart.assign(nKF + 1, 0); hs.peList.resize(nE);
    for (int s = 0; s < nE; s++) hs.peStart[H.h_eKF[s] + 1]++;
    for (int k = 0; k < nKF; k++) hs.peStart[k + 1] += hs.peStart[k];
    hs.fill.assign(hs.peStart.begin(), hs.peStart.end() - 1);
    for (int s = 0; s < nE; s++) hs.peList[hs.fill[H.h_eKF[s]]++] = s;
    std::vector<Pose> poses(nKF);
    for (int k = 0; k < nKF; k++) poses[k] = pose_from_Tcw32(p->Tcw + 16 * k);
    H.fixed.assign(p->kf_fixed, p->kf_fixed + nKF); H.level.assign(nE, 0); H.poseIdx.assign(nKF, -1); H.ptAct.assign(nMP, 0);
    std::vector<int> kfOfQ;
    for (int k = 0; k < nKF; k++) if (!H.fixed[k]) kfOfQ.push_back(k);
    const int nQ = (int)kfOfQ.size();
    D.nQ = nQ;
    int rc;
    const int nmax = 6 * nQ;
    const auto tp1 = tNow();
    const Pose* cpose = nullptr; double* cX = nullptr;
    int* d_eMP = nullptr; int* d_eKF = nullptr; int* d_perm = nullptr; float2* d_kp = nullptr; float* d_isig = nullptr; float* d_pts32 = nullptr; int* d_bad = nullptr;
    double* d_obs = nullptr; int8_t* d_face = nullptr;
    if ((rc = dupload(o, &cpose, poses)) || (rc = dupload(o, &D.lmStart, hs.lmStart)) || (rc = dupload(o, &D.peStart, hs.peStart)) || (rc = dupload(o, &D.peList, hs.peList)) ||
        (rc = dupload(o, &D.kfOfQ, kfOfQ)) || (rc = dalloc(o, &d_eMP, nE)) || (rc = dalloc(o, &d_eKF, nE)) || (rc = dalloc(o, &d_kp, nEg)) || (rc = dalloc(o, &d_isig, nEg)) ||
        (rc = dalloc(o, &d_pts32, (size_t)nMP * 3)) || (rc = dalloc(o, &cX, (size_t)nMP * 3)) || (rc = dalloc(o, &d_obs, (size_t)nE * 3)) || (rc = dalloc(o, &d_face, nE)) ||
        (rc = dalloc(o, &d_bad, 1)) || (!grouped && (rc = dalloc(o, &d_perm, nE)))) return rc;
    if (nE > 0) {
        CSLAM_CUDA(cudaMemcpyAsync(d_eMP, H.h_eMP, (size_t)nE * 4, cudaMemcpyHostToDevice, o->stream));
        CSLAM_CUDA(cudaMemcpyAsync(d_eKF, H.h_eKF, (size_t)nE * 4, cudaMemcpyHostToDevice, o->stream));
        CSLAM_CUDA(cudaMemcpyAsync(d_kp, p->kp_xy, (size_t)nEg * 8, cudaMemcpyHostToDevice, o->stream));
        CSLAM_CUDA(cudaMemcpyAsync(d_isig, p->inv_sigma2, (size_t)nEg * 4, cudaMemcpyHostToDevice, o->stream));
        if (!grouped) CSLAM_CUDA(cudaMemcpyAsync(d_perm, H.perm, (size_t)nE * 4, cudaMemcpyHostToDevice, o->stream));
    }
    if (nMP > 0) CSLAM_CUDA(cudaMemcpyAsync(d_pts32, p->points, (size_t)nMP * 12, cudaMemcpyHostToDevice, o->stream));
    CSLAM_CUDA(cudaMemsetAsync(d_bad, 0x7f, sizeof(int), o->stream));
    if (nE > 0) { k_ba_prep_edges<<<cdiv(nE, 256), 256, 0, o->stream>>>(nE, d_perm, d_kp, d_isig, p->face_w, p->face_h, d_obs, d_face, d_bad); o->launches++; }
    if (nMP > 0) { k_ba_prep_points<<<cdiv(nMP * 3, 256), 256, 0, o->stream>>>(nMP * 3, d_pts32, cX); o->launches++; }
    D.eMP = d_eMP; D.eKF = d_eKF; D.obs = d_obs; D.face = d_face;
    D.pose = const_cast<Pose*>(cpose); D.X = cX;
    H.ldp = ((nmax + 1 + 8) + 3) & ~3;
    const size_t payloadMax = (size_t)nmax * nmax + 2 * (size_t)nmax + 4;
    const int maxBlocks = std::max({cdiv(nE, 256), cdiv(nmax + 3 * nMP, 256), 1});
    long long* pairCnt = nullptr;
    if ((rc = dalloc(o, &D.poseBak, nKF)) || (rc = dalloc(o, &D.Xbak, (size_t)nMP * 3)) || (rc = dalloc(o, &D.err, (size_t)nE * 2, true)) || (rc = dalloc(o, &D.level, nE, true)) ||
        (rc = dalloc(o, &H.d_poseIdx, nKF)) || (rc = dalloc(o, &H.d_pact, nKF + 1)) || (rc = dalloc(o, &H.d_ptAct, nMP)) || (rc = dalloc(o, &H.d_flag, nE)) || (rc = dalloc(o, &D.Hpp, (size_t)std::max(nQ, 1) * 36)) ||
        (rc = dalloc(o, &D.bp, (size_t)std::max(nQ, 1) * 6)) || (rc = dalloc(o, &D.Hll, (size_t)nMP * 9)) || (rc = dalloc(o, &D.bl, (size_t)nMP * 3)) ||
        (rc = dalloc(o, &D.Hpl, (size_t)nE * 18)) || (rc = dalloc(o, &D.Dinv, (size_t)nMP * DINV_LD)) || (rc = dalloc(o, &D.db, (size_t)nMP * 3)) ||
        (rc = dalloc(o, &H.red, payloadMax)) || (rc = dalloc(o, &D.xp, std::max(nmax, 1), true)) || (rc = dalloc(o, &D.xl, (size_t)nMP * 3, true)) ||
        (rc = dalloc(o, &D.scal, 8, true)) || (rc = dalloc(o, &D.part, maxBlocks)) || (rc = dalloc(o, &D.ticket, 4, true)) || (rc = dalloc(o, &D.posePart, (size_t)std::max(nQ, 1) * POSE_SPLIT * 27)) || (rc = dalloc(o, &D.poseTicket, std::max(nQ, 1), true)) ||
        (rc = dalloc(o, &H.Lt, (size_t)LD_NB * H.ldp)) || (rc = dalloc(o, &H.LDt, (size_t)LD_NB * H.ldp)) || (rc = dalloc(o, &H.Minv, (size_t)(nmax / LD_NB + 1) * LD_NB * LD_NB)) || (rc = dalloc(o, &pairCnt, (size_t)nQ * nQ + 1)) ||
        (rc = dalloc(o, &H.d_xerr, 1, true))) return rc;
    D.poseIdx = H.d_poseIdx; D.ptAct = H.d_ptAct;
    if (getenv("CSLAM_BA_PROFILE")) { if ((rc = dalloc(o, &H.d_prof, 8, true))) return rc; }
    // ---- multi-GPU exchange path
    if (o->nranks > 1) {
        if (!getenv("CSLAM_BA_NCCL_ONLY") && (!o->oneShot || o->xchgBytes < payloadMax * 8)) {
            const int xr = setup_xchg(o, payloadMax * 8);
            if (xr < 0) return xr;
        }
        H.useOneShot = o->oneShot && o->xchgBytes >= payloadMax * 8 && !getenv("CSLAM_BA_NCCL_ONLY");
        H.xstride = ((o->xchgBytes + 255) & ~(size_t)255) / 8;
        if ((rc = dalloc(o, &H.HppFull, (size_t)std::max(nQ, 1) * 36))) return rc;
    }
    // ---- co-observation lists (once per call, all edges)
    int badEdge = 0x7f7f7f7f;
    if (nQ > 0) {
        k_ba_pairs_count<<<dim3(nQ, nQ), 128, 0, o->stream>>>(D, pairCnt); o->launches++;
        k_ba_pairs_scan<<<1, 1024, 0, o->stream>>>(pairCnt, nQ * nQ); o->launches++;
        long long total = 0;
        CSLAM_CUDA(cudaMemcpyAsync(&total, pairCnt + (size_t)nQ * nQ, sizeof(long long), cudaMemcpyDeviceToHost, o->stream));
        CSLAM_CUDA(cudaMemcpyAsync(&badEdge, d_bad, sizeof(int), cudaMemcpyDeviceToHost, o->stream));
        CSLAM_CUDA(cudaStreamSynchronize(o->stream));
        if (badEdge < nEg) { set_error("edge %d: keypoint (%g,%g) is on no cube face (the reference calls exit() here)", badEdge, p->kp_xy[2 * badEdge], p->kp_xy[2 * badEdge + 1]); return CSLAM_E_BADARG; }
        int4* tuples = nullptr;
        if ((rc = dalloc(o, &tuples, (size_t)std::max<long long>(total, 1)))) return rc;
        k_ba_pairs_fill<<<dim3(nQ, nQ), 128, 0, o->stream>>>(D, pairCnt, tuples); o->launches++;
        CSLAM_CUDA(cudaGetLastError());
        D.pairStart = pairCnt; D.tuples = tuples;
    }
    if (nQ == 0) {
        CSLAM_CUDA(cudaMemcpyAsync(&badEdge, d_bad, sizeof(int), cudaMemcpyDeviceToHost, o->stream));
        CSLAM_CUDA(cudaStreamSynchronize(o->stream));
        if (badEdge < nEg) { set_error("edge %d: keypoint (%g,%g) is on no cube face (the reference calls exit() here)", badEdge, p->kp_xy[2 * badEdge], p->kp_xy[2 * badEdge + 1]); return CSLAM_E_BADARG; }
    }
    if (hostProf) cudaStreamSynchronize(o->stream);
    const auto tp2 = tNow();
    // ---- src/Optimizer.cpp:363-395
    if ((rc = H.initialize())) return rc;
    if ((rc = H.optimize(its1))) return rc;
    std::vector<uint8_t> flags;
    if (!H.terminate()) {
        if ((rc = H.classify(flags))) return rc;
        for (int s = 0; s < nE; s++) if (flags[s]) H.level[s] = 1;
        D.robust = 0;
        if ((rc = H.initialize())) return rc;
        if ((rc = H.optimize(its2))) return rc;
    }
    if ((rc = H.classify(flags))) return rc;
    std::vector<uint8_t> gflags;   // multi-GPU: every rank returns the flags of ALL edges (max over the owners' flags, in the caller's order)
    if (multi) {
        uint8_t* d_gflag = nullptr;
        if ((rc = dalloc(o, &d_gflag, std::max(nEg, 1), true))) return rc;
        if (nE > 0) { k_ba_scatter_flags<<<cdiv(nE, 256), 256, 0, o->stream>>>(nE, d_perm, H.d_flag, d_gflag); o->launches++; }
        rc = nccl_api()->AllReduce(d_gflag, d_gflag, nEg, NCCL_U8, NCCL_MAX, o->comm, o->stream);
        if (rc) { set_error("ncclAllReduce (flags) failed (%d)", rc); return CSLAM_E_NCCL; }
        gflags.resize(nEg);
        CSLAM_CUDA(cudaMemcpyAsync(gflags.data(), d_gflag, nEg, cudaMemcpyDeviceToHost, o->stream));
        CSLAM_CUDA(cudaStreamSynchronize(o->stream));
    }
    const auto tp3 = tNow();
    H.drop_graph();
    if (H.d_prof) {
        long long hp[8]; cudaMemcpyAsync(hp, H.d_prof, sizeof(hp), cudaMemcpyDeviceToHost, o->stream); cudaStreamSynchronize(o->stream);
        static const char* nm[8] = {"load diag", "factor diag", "trsm", "cluster sync 1", "stage panel", "trailing update", "cluster sync 2", "back substitution"};
        for (int k = 0; k < 8; k++) std::fprintf(stderr, "[k_ba_solve] %-18s %10.1f kclk total, %7.2f us per trial\n", nm[k], hp[k] / 1e3, hp[k] / 1.9e3 / std::max(H.trials, 1));
    }
    // ---- write back (src/Optimizer.cpp:432-450): float32 poses / points; with landmark sharding every rank holds its own points
    if (o->nranks > 1) {
        k_ba_mask_points<<<H.grid(nMP), 256, 0, o->stream>>>(D); o->launches++;
        if ((rc = H.allreduce(D.X, (size_t)nMP * 3, NCCL_SUM))) return rc;
    }
    CSLAM_CUDA(cudaMemcpyAsync(poses.data(), D.pose, nKF * sizeof(Pose), cudaMemcpyDeviceToHost, o->stream));
    hs.X.resize((size_t)nMP * 3);
    std::vector<double>& X = hs.X;
    CSLAM_CUDA(cudaMemcpyAsync(X.data(), D.X, X.size() * 8, cudaMemcpyDeviceToHost, o->stream));
    CSLAM_CUDA(cudaStreamSynchronize(o->stream));
    for (int k = 0; k < nKF; k++) {
        pose_to_Tcw32(poses[k], p->Tcw + 16 * k);
        if (r && r->pose_fp64) { double* q = r->pose_fp64 + 7 * k; q[0] = poses[k].t[0]; q[1] = poses[k].t[1]; q[2] = poses[k].t[2]; q[3] = poses[k].q[0]; q[4] = poses[k].q[1]; q[5] = poses[k].q[2]; q[6] = poses[k].q[3]; }
    }
    for (size_t i = 0; i < X.size(); i++) { p->points[i] = (float)X[i]; if (r && r->points_fp64) r->points_fp64[i] = X[i]; }
    if (r) {
        if (r->outlier) { if (multi) std::memcpy(r->outlier, gflags.data(), nEg); else for (int s = 0; s < nE; s++) r->outlier[H.perm ? H.perm[s] : s] = flags[s]; }
        r->iterations = H.iterations; r->trials = H.trials;
    }
    free_pool(o);
    if (hostProf) std::fprintf(stderr, "[cslam_local_ba] host prep %.3f ms, upload + co-observation lists %.3f ms, LM schedule %.3f ms (%d trials), write-back %.3f ms\n", tMs(tp0, tp1), tMs(tp1, tp2), tMs(tp2, tp3), H.trials, tMs(tp3, tNow()));
    return CSLAM_OK;
}
