"""GPU parity of the device tracking chain (configs[4], the per-frame Tracking loop): k_gather_pose_inputs against gather_ref bit for bit,
k_pose_opt at tracking size against the fp64 oracle, the strided cslam_pose_optimization_dev against the host entry, and the whole
frame index -> SearchByProjection(last frame) -> gather -> PoseOptimization chain on device buffers against the CPU chain.

Pose gates are test_gpu_ba.py's: 1e-5 relative on the fp64 pose (host entry only; the device entry returns float32 Tcw), Tcw within 2e-6,
equal inlier counts and equal outlier vectors. pose_optimization_dev returns outlier flags in gathered (compacted) order."""
import numpy as np
import pytest

from cubemapslam_b200 import config, synth

from . import tracking_chain_ref as R

pytestmark = pytest.mark.gpu
RTOL = 1e-5
SENT32 = np.uint32(0x7FC0DEAD)      # a NaN payload no kernel computes
NCELLS = 5 * 50 * 50


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


@pytest.fixture(scope="module")
def opt():
    from cubemapslam_b200.optimizer import Optimizer
    o = Optimizer()
    yield o
    o.close()


@pytest.fixture(scope="module")
def trk():
    from cubemapslam_b200.tracker import Tracker
    t = Tracker(max_frames=1, max_features=64)     # the device entries only use its stream and capacity flag
    yield t
    t.close()


def rel(a, b):
    return np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-30)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _kp_bytes(k):
    return np.ascontiguousarray(k, R.KP_DTYPE).view(np.uint8).reshape(k.shape + (28,))


def _kp_host(t):
    return np.ascontiguousarray(t.cpu().numpy()).view(R.KP_DTYPE)[..., 0]


# ------------------------------------------------------------------------------------------------- k_gather_pose_inputs
GATHER_N = [0, 1, 31, 32, 33, 255, 256, 257, 511, 513, 4096]


def test_gather_pose_inputs_bit_exact(torch, trk):
    cs, ls = 4096, 3001
    n = np.array(GATHER_N + [5000], np.int32)          # the last frame claims more key points than its row holds: clamped to cs
    P = len(n)
    rng = np.random.default_rng(17)
    cth = R.cos_fov_th(config.front_1024()["Camera.fov"])
    isg = R.inv_sigma2_levels()
    k = np.zeros((P, cs), R.KP_DTYPE)
    k["x"] = rng.uniform(0, 1950, (P, cs)); k["y"] = rng.uniform(0, 1950, (P, cs)); k["octave"] = rng.integers(0, 8, (P, cs))
    match = rng.integers(0, ls, (P, cs)).astype(np.int32)          # slots past n[p] keep valid-looking indices: they must be ignored
    sel = rng.random((P, cs))
    match[sel < 0.3] = -1; match[(sel >= 0.3) & (sel < 0.45)] = -2
    match[-1, cs - 1] = ls - 1; match[-2, 4095] = ls - 1              # the last valid index of the last frames' rows
    rays = rng.uniform(-1, 1, (P, cs, 3)).astype(np.float32)
    planted = [cth, np.nextafter(cth, np.float32(-np.inf)), np.float32(0), np.float32(np.nan)]
    for p in range(P):
        m = min(n[p], cs)
        for j, z in enumerate(planted):
            if j < m:
                i = (j * 97 + p) % m
                rays[p, i, 2] = z
                match[p, i] = (p * 13 + j) % ls
    XwL = rng.normal(0, 5, (P, ls, 3)).astype(np.float32)
    d_match, d_k, d_n, d_rays, d_X, d_isg = (_dev(torch, a) for a in (match, _kp_bytes(k), n, rays, XwL, isg))
    ts = torch.cuda.ExternalStream(trk.stream)
    for use_rays in (True, False):
        outX, outK, outW = (_dev(torch, np.full(shape, SENT32, np.uint32).view(np.float32)) for shape in ((P, cs, 3), (P, cs, 2), (P, cs)))
        cnt = _dev(torch, np.full(P, -7, np.int32))
        ts.wait_stream(torch.cuda.current_stream())
        trk.gather_pose_inputs_dev(P, d_match.data_ptr(), d_k.data_ptr(), d_n.data_ptr(), cs, d_rays.data_ptr() if use_rays else None, cth, d_X.data_ptr(), ls,
                                   d_isg.data_ptr(), outX.data_ptr(), outK.data_ptr(), outW.data_ptr(), cnt.data_ptr())
        trk.sync()
        gX, gK, gW = (bits(t.cpu().numpy()) for t in (outX, outK, outW)); gc = cnt.cpu().numpy()
        dropped = 0
        for p in range(P):
            Xr, kr, wr, c = R.gather_ref(match[p], k[p], n[p], cs, rays[p] if use_rays else None, cth, XwL[p], isg)
            assert gc[p] == c, (use_rays, p, gc[p], c)
            assert np.array_equal(gX[p, :c], bits(Xr)) and np.array_equal(gK[p, :c], bits(kr)) and np.array_equal(gW[p, :c], bits(wr)), (use_rays, p)
            assert np.all(gX[p, c:] == SENT32) and np.all(gK[p, c:] == SENT32) and np.all(gW[p, c:] == SENT32), (use_rays, p)
            dropped += int(np.count_nonzero(match[p, :min(n[p], cs)] >= 0)) - c
        assert (dropped > 0) == use_rays


# ------------------------------------------------------------------------------------------------- k_pose_opt at tracking size
POSE_N = [3, 9, 10, 11, 255, 256, 257, 513, 1500, 3000, 4096]
FRACS = [0.0, 0.15, 0.5]
REPS = 5


def _pose_frames(W):
    """REPS copies of every (size, outlier fraction) in a shuffled order, plus frames of 0, 1 and 2 correspondences first, in the middle and last."""
    frames = []
    for r in range(REPS):
        for nn in POSE_N:
            for fr in FRACS:
                frames.append(R.pose_case(nn, faceW=W, seed=r % 2, outlier_frac=fr, offset=(r * 389) % (4097 - nn)))
    order = np.random.default_rng(W).permutation(len(frames))
    frames = [frames[i] for i in order]
    frames.insert(0, R.pose_case(0, faceW=W)); frames.insert(len(frames) // 2, R.pose_case(1, faceW=W, offset=7)); frames.append(R.pose_case(2, faceW=W, offset=11))
    return frames


def _host_batch(opt, frames, W):
    off = np.cumsum([0] + [len(q["Xw"]) for q in frames]).astype(np.int32)
    T = np.stack([q["Tcw"] for q in frames])
    g = opt.PoseOptimization(T, np.concatenate([q["Xw"] for q in frames]), np.concatenate([q["kpxy"] for q in frames]),
                             np.concatenate([q["inv_sigma2"] for q in frames]), W, W, offset=off)
    return g, off


def _check_host_vs_oracle(oracle, opt, frames, W, worst=None):
    g, off = _host_batch(opt, frames, W)
    refs = []
    for i, q in enumerate(frames):
        r = oracle.pose_opt(q["Tcw"], q["Xw"], q["kpxy"], q["inv_sigma2"], W, W)
        refs.append(r)
        n = len(q["Xw"])
        assert g["inliers"][i] == r["inliers"], (i, n, g["inliers"][i], r["inliers"])
        assert np.array_equal(g["outlier"][off[i]:off[i + 1]], r["outlier"]), (i, n)
        if n >= 3:
            e = rel(g["pose64"][i], r["pose64"])
            assert e < RTOL, (i, n, e)
            assert np.allclose(g["Tcw"][i], r["Tcw"], rtol=0, atol=2e-6), (i, n)
            if worst is not None:
                worst[n] = max(worst.get(n, 0.0), e)
        else:
            assert g["inliers"][i] == 0 and np.array_equal(bits(g["Tcw"][i]), bits(q["Tcw"])), (i, n)   # untouched (src/Optimizer.cpp:133-134)
    return g, off, refs


@pytest.mark.parametrize("W", [650, 450])
def test_pose_optimization_tracking_sizes(oracle, opt, W):
    frames = _pose_frames(W)
    assert len(frames) > 148                                              # more CTAs than the B200 has SMs
    worst = {}
    _check_host_vs_oracle(oracle, opt, frames, W, worst)
    print("\nk_pose_opt vs oracle, face %d: worst pose64 relative error per size: %s" % (W, ", ".join("%d: %.1e" % kv for kv in sorted(worst.items()))))


def _scrambled(W):
    q = R.pose_case(300, faceW=W, seed=3, outlier_frac=0.15)
    q["kpxy"] = q["kpxy"][np.random.default_rng(0).permutation(300)]
    return q


def _at_camera_centre(W):
    q = R.pose_case(300, faceW=W, seed=3, outlier_frac=0.15)
    T = q["Tcw"].astype(np.float64)
    q["Xw"][5] = (-T[:3, :3].T @ T[:3, 3]).astype(np.float32)
    return q


def _on_tile_boundaries(W):
    """Per face, the observations nearest the tile's left and top edges moved exactly onto them (x = c*W, y = r*W)."""
    q = R.pose_case(1500, faceW=W, seed=4, outlier_frac=0.15)
    kp = q["kpxy"]
    for c, r in synth._FACE_TILE.values():
        on = np.nonzero(_in_tile(kp, c, r, W))[0]
        for axis, edge in ((0, c * W), (1, r * W)):
            near = on[np.argsort(kp[on, axis] - edge)[:3]]
            kp[near, axis] = np.float32(edge)
    return q


def _in_tile(kp, c, r, W):
    return (kp[:, 0] >= c * W) & (kp[:, 0] < (c + 1) * W) & (kp[:, 1] >= r * W) & (kp[:, 1] < (r + 1) * W)


@pytest.mark.parametrize("W", [650, 450])
def test_pose_optimization_edge_cases(oracle, opt, W):
    frames = [_scrambled(W), _at_camera_centre(W), R.pose_case(600, faceW=W, seed=2, outlier_frac=0.15, rot=0.05, trans=0.02), _on_tile_boundaries(W)]
    g, off, refs = _check_host_vs_oracle(oracle, opt, frames, W)
    sc, cc, big, tb = refs
    # scrambled: round 0 (all 300 edges, chi2 ~1e6) leaves one edge active; rounds 1 and 2 fit it alone (rank-2 H, identical logs);
    # round 3 has no active edge (nAct == 0) and logs nothing
    L = sc["log"]
    assert sc["inliers"] <= 3 and len(L) == 13, L
    assert np.all(L[:7, 0] > 1e5) and np.all(L[7:, 0] < 1e-6) and np.array_equal(L[7:10], L[10:13]), L
    assert cc["log"][0, 1] > 1e12 and cc["inliers"] > 100                 # lambda starts at 2.5e12 (450 px) / 3.5e12 (650 px); the pose barely moves
    assert big["log"][:, 2].max() > 1                                     # rejected trials
    kp = frames[3]["kpxy"]
    for c, r in synth._FACE_TILE.values():                                # planted on every face, inside that face's tile
        t = _in_tile(kp, c, r, W)
        assert np.any(kp[t, 0] == c * W) and np.any(kp[t, 1] == r * W), (c, r)


def test_pose_optimization_robust_switch_round(oracle, opt):
    """The robust kernel is on for rounds 0-2 and off for round 3. Round 3 restarts from the prior with the active set that round 2's
    classification left, so a wrong switch round only shows when round 2's robust and plain trajectories classify some edge differently.
    Observation 7 is planted 2.47428 px off its exact projection (chi2 just at 5.991) so that they do: an oracle that turns the robust kernel
    off one round early returns 258 inliers here instead of 259 and a pose 7.5e-5 (relative) away. The window that separates the two is
    one float32 key-point coordinate wide; other frames of this suite do not tell the two schedules apart."""
    W = 650
    q = R.plant_observation(R.pose_case(300, faceW=W, seed=1, outlier_frac=0.15, rot=0.1, trans=0.05), 7, 2.47428)
    _, _, (r,) = _check_host_vs_oracle(oracle, opt, [q], W)
    assert r["inliers"] == 259


# ------------------------------------------------------------------------------------------------- cslam_pose_optimization_dev addressing
def test_pose_optimization_dev_matches_host_entry(torch, opt):
    W, S = 650, 4096
    frames = _pose_frames(W)
    g, off = _host_batch(opt, frames, W)
    F = len(frames)
    cnt = np.array([len(q["Xw"]) for q in frames], np.int32)
    over = int(np.nonzero(cnt == S)[0][0]); cnt[over] = 5000                 # count > stride reads as count = stride
    rng = np.random.default_rng(3)
    Xw = np.full((F, S, 3), np.nan, np.float32); kp = rng.uniform(0, 3 * W, (F, S, 2)).astype(np.float32); w = np.full((F, S), np.nan, np.float32)
    for i, q in enumerate(frames):                                        # the tail of every row is poison: it must never be read
        m = len(q["Xw"]); Xw[i, :m] = q["Xw"]; kp[i, :m] = q["kpxy"]; w[i, :m] = q["inv_sigma2"]
    T0 = np.stack([q["Tcw"] for q in frames])
    d_T, d_X, d_kp, d_w, d_c = (_dev(torch, a) for a in (T0, Xw, kp, w, cnt))
    d_out = _dev(torch, np.full((F, S), 0xAB, np.uint8)); d_inl = _dev(torch, np.full(F, -7, np.int32))
    os_ = torch.cuda.ExternalStream(opt.stream)
    os_.wait_stream(torch.cuda.current_stream())
    opt.pose_optimization_dev(F, S, d_c.data_ptr(), d_T.data_ptr(), d_X.data_ptr(), d_kp.data_ptr(), d_w.data_ptr(), W, W, d_out.data_ptr(), d_inl.data_ptr())
    opt.sync()
    T, out, inl = d_T.cpu().numpy(), d_out.cpu().numpy(), d_inl.cpu().numpy()
    assert np.array_equal(inl, g["inliers"])
    for i, q in enumerate(frames):
        m = len(q["Xw"])
        assert np.array_equal(bits(T[i]), bits(g["Tcw"][i])), i            # the host entry leaves n < 3 frames untouched too
        if m < 3:
            assert inl[i] == 0 and np.array_equal(bits(T[i]), bits(T0[i])), i
        assert np.array_equal(out[i, :m], g["outlier"][off[i]:off[i + 1]]), i
        assert np.all(out[i, m:] == 0xAB), i
    assert {len(frames[i]["Xw"]) for i in range(F) if len(frames[i]["Xw"]) < 3} == {0, 1, 2}


# ------------------------------------------------------------------------------------------------- the chain end to end
class _Chain:
    """Device buffers of one batch of (last, current) frames and the four launches of the bench's tracking pass, ordered on the tracker's and
    the optimizer's streams like bench_extra._tracking_leg."""

    def __init__(self, torch, P, cs, ls):
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device="cuda")
        u8, i32, f32 = torch.uint8, torch.int32, torch.float32
        self.torch, self.P, self.cs, self.ls = torch, P, cs, ls
        self.rays = z((P, cs, 3), f32); self.cellStart = z((P, NCELLS + 1), torch.int16); self.cellIdx = z((P, cs), torch.int16)
        self.match = z((P, cs), i32); self.nm = z((P,), i32)
        self.gX = z((P, cs, 3), f32); self.gK = z((P, cs, 2), f32); self.gW = z((P, cs), f32); self.count = z((P,), i32)
        self.outl = z((P, cs), u8); self.inl = z((P,), i32)
        self.isg = _dev(torch, R.inv_sigma2_levels())

    def run(self, trk, opt, kC, dC, nC, taken, Tcw, kL, nL, has, Xw, dL, obs, cth, th=15.0, check_ori=True, index=True):
        torch, P, cs, ls = self.torch, self.P, self.cs, self.ls
        ts = torch.cuda.ExternalStream(trk.stream); os_ = torch.cuda.ExternalStream(opt.stream)
        ts.wait_stream(torch.cuda.current_stream())
        if index:
            trk.frame_index_dev(kC.data_ptr(), nC.data_ptr(), P, cs, 650, 650, self.rays.data_ptr(), self.cellStart.data_ptr(), self.cellIdx.data_ptr())
        trk.search_by_projection_last_dev(P, kC.data_ptr(), dC.data_ptr(), nC.data_ptr(), cs, self.cellStart.data_ptr(), self.cellIdx.data_ptr(), taken.data_ptr(), Tcw.data_ptr(),
                                          kL.data_ptr(), nL.data_ptr(), ls, has.data_ptr(), Xw.data_ptr(), dL.data_ptr(), obs.data_ptr(), 650, 650, cth, th, int(check_ori),
                                          self.match.data_ptr(), self.nm.data_ptr())
        trk.gather_pose_inputs_dev(P, self.match.data_ptr(), kC.data_ptr(), nC.data_ptr(), cs, self.rays.data_ptr(), cth, Xw.data_ptr(), ls, self.isg.data_ptr(),
                                   self.gX.data_ptr(), self.gK.data_ptr(), self.gW.data_ptr(), self.count.data_ptr())
        os_.wait_stream(ts)
        opt.pose_optimization_dev(P, cs, self.count.data_ptr(), Tcw.data_ptr(), self.gX.data_ptr(), self.gK.data_ptr(), self.gW.data_ptr(), 650, 650, self.outl.data_ptr(),
                                  self.inl.data_ptr())
        opt.sync()
        trk.sync()                                                         # also raises if a search window overflowed its capacity
        return {k: getattr(self, k).cpu().numpy() for k in ("rays", "cellStart", "cellIdx", "match", "nm", "gX", "gK", "gW", "count", "outl", "inl")}


def _check_task(oracle, s, g, p, nC, cth, T_after, ref=None):
    """Every stage of task p against the CPU chain; returns the oracle chain."""
    kCur = s["kCur"]
    r_rays, _ = oracle.key_point_rays(kCur, 650, 650)
    assert np.array_equal(bits(g["rays"][p, :nC]), bits(r_rays)), p
    start, idx = oracle.FrameGrid(kCur, 650, 650).csr()
    assert np.array_equal(g["cellStart"][p].view(np.uint16).astype(np.int32), start) and np.array_equal(g["cellIdx"][p, :nC].view(np.uint16).astype(np.int32), idx), p
    c = R.oracle_chain(oracle, s, cth) if ref is None else ref
    m = g["match"][p, :nC]
    assert g["nm"][p] == c["nmatches"] and np.array_equal(np.where(m == -2, -1, m), c["match"]), p
    Xr, kr, wr, cnt = R.gather_ref(g["match"][p], kCur, nC, len(g["match"][p]), g["rays"][p], cth, s["Xw"], R.inv_sigma2_levels())
    assert g["count"][p] == cnt == c["count"], p
    assert np.array_equal(bits(g["gX"][p, :cnt]), bits(Xr)) and np.array_equal(bits(g["gK"][p, :cnt]), bits(kr)) and np.array_equal(bits(g["gW"][p, :cnt]), bits(wr)), p
    assert np.array_equal(bits(Xr), bits(c["Xw"])) and np.array_equal(bits(kr), bits(c["kp"])), p
    po = c["pose"]
    assert g["inl"][p] == po["inliers"], (p, g["inl"][p], po["inliers"])
    assert np.array_equal(g["outl"][p, :cnt], po["outlier"]), p            # gathered order
    assert np.allclose(T_after[p], po["Tcw"], rtol=0, atol=2e-6), p
    return c


def test_chain_planted_tasks(oracle, torch, trk, opt):
    sizes = [3000, 1200, 2200, 3500, 400, 2800]
    tasks = [R.tracking_task(40 + i, n=n) for i, n in enumerate(sizes)]
    tasks[1]["mpObs"][:] = 0                                               # no MapPoint has observations: taken slots stay free
    tasks[4]["curTaken"][::4] = 1
    P = len(tasks)
    cs = max(len(s["kCur"]) for s in tasks) + 5; ls = max(sizes) + 3
    assert cs <= 4096 and cs != ls
    kC = np.zeros((P, cs), R.KP_DTYPE); dC = np.zeros((P, cs, 32), np.uint8); tk = np.zeros((P, cs), np.uint8); nC = np.zeros(P, np.int32)
    kL = np.zeros((P, ls), R.KP_DTYPE); has = np.zeros((P, ls), np.uint8); Xw = np.zeros((P, ls, 3), np.float32); dL = np.zeros((P, ls, 32), np.uint8)
    ob = np.zeros((P, ls), np.uint8); nL = np.zeros(P, np.int32)
    for i, s in enumerate(tasks):
        a, b = len(s["kCur"]), len(s["kLast"]); nC[i] = a; nL[i] = b
        kC[i, :a] = s["kCur"]; dC[i, :a] = s["dCur"]; tk[i, :a] = s["curTaken"]
        kL[i, :b] = s["kLast"]; has[i, :b] = s["hasMP"]; Xw[i, :b] = s["Xw"]; dL[i, :b] = s["dLast"]; ob[i, :b] = s["mpObs"] > 0
    T0 = np.stack([s["Tcw"] for s in tasks])
    d = [_dev(torch, a) for a in (_kp_bytes(kC), dC, nC, tk, T0, _kp_bytes(kL), nL, has, Xw, dL, ob)]
    cth = R.cos_fov_th(config.front_1024()["Camera.fov"])
    ch = _Chain(torch, P, cs, ls)
    g = ch.run(trk, opt, *d, cth)
    T = d[4].cpu().numpy()
    assert np.count_nonzero(g["match"] == -2) > 0                          # the rotation check cleared slots
    for p, s in enumerate(tasks):
        c = _check_task(oracle, s, g, p, nC[p], cth, T)
        assert np.all(s["src"][c["match"] >= 0] == c["match"][c["match"] >= 0]), p
        a0, t0 = R.pose_errors(s["Tcw"], s["Ttrue"]); a1, t1 = R.pose_errors(T[p], s["Ttrue"])
        print("\nplanted task %d: %d matches, %d gathered, %d inliers; prior %.1e rad / %.1e, result %.1e rad / %.1e"
              % (p, g["nm"][p], g["count"][p], g["inl"][p], a0, t0, a1, t1))
        if g["count"][p] > 100:
            assert t1 < 0.5 * t0 and a1 < a0, p


def test_chain_extracted_frames(oracle, torch, trk, opt):
    from cubemapslam_b200.frontend import FrontEnd
    cfg = config.front_1024(); mask = config.load_mask("gray_cubemap_front_mask_650")
    P = 5
    last = np.stack([synth.fisheye_frame(cfg, i) for i in range(P)])
    cur = np.roll(last, 7, axis=2); cur[P - 1] = 0                          # the last task's current frame is all black: no key points
    fe = FrontEnd(cfg, mask, max_batch=2 * P)
    cap = fe.kp_cap
    fish = _dev(torch, np.concatenate([last, cur]))
    u8 = torch.uint8
    kps = torch.zeros((2 * P, cap, 28), dtype=u8, device="cuda"); desc = torch.zeros((2 * P, cap, 32), dtype=u8, device="cuda"); nout = torch.zeros(2 * P, dtype=torch.int32, device="cuda")
    fs = torch.cuda.ExternalStream(fe.stream)
    fs.wait_stream(torch.cuda.current_stream())
    fe.run_dev(fish.data_ptr(), 2 * P, kps.data_ptr(), desc.data_ptr(), nout.data_ptr()); fe.sync()
    # the last frames' rays give the MapPoints (depth 4 along the ray, world = last camera), as in the bench
    rays = torch.zeros((P, cap, 3), dtype=torch.float32, device="cuda"); cellStart = torch.zeros((P, NCELLS + 1), dtype=torch.int16, device="cuda")
    cellIdx = torch.zeros((P, cap), dtype=torch.int16, device="cuda")
    ts = torch.cuda.ExternalStream(trk.stream); ts.wait_stream(fs)
    trk.frame_index_dev(kps.data_ptr(), nout.data_ptr(), P, cap, 650, 650, rays.data_ptr(), cellStart.data_ptr(), cellIdx.data_ptr()); trk.sync()
    Xw = (rays * 4.0).contiguous()
    nL = nout[:P].contiguous(); nC = nout[P:].contiguous()
    has = (torch.arange(cap, device="cuda")[None, :] < nL[:, None]).to(u8).contiguous(); obs = torch.ones_like(has); taken = torch.zeros((P, cap), dtype=u8, device="cuda")
    T0 = np.tile(np.eye(4, dtype=np.float32), (P, 1, 1)); T0[:, 0, 3] = 0.01
    d_T = _dev(torch, T0)
    kC = kps[P:].contiguous(); dC = desc[P:].contiguous()
    cth = R.cos_fov_th(cfg["Camera.fov"])
    ch = _Chain(torch, P, cap, cap)
    g = ch.run(trk, opt, kC, dC, nC, taken, d_T, kps[:P].contiguous(), nL, has, Xw, desc[:P].contiguous(), obs, cth)
    fe.close()
    T = d_T.cpu().numpy(); hk = _kp_host(kps); hd = desc.cpu().numpy(); hn = nout.cpu().numpy(); hX = Xw.cpu().numpy(); hr = rays.cpu().numpy()
    assert hn[2 * P - 1] == 0 and g["nm"][P - 1] == 0 and g["count"][P - 1] == 0 and g["inl"][P - 1] == 0
    assert np.array_equal(bits(T[P - 1]), bits(T0[P - 1]))                 # fewer than 3 correspondences: Tcw untouched
    sc = R.scale_factors()
    for p in range(P - 1):
        a, b = hn[P + p], hn[p]
        assert a > 1000 and b > 1000, (p, a, b)
        r_last, _ = oracle.key_point_rays(hk[p, :b], 650, 650)
        assert np.array_equal(bits(hr[p, :b]), bits(r_last)), p
        s = dict(kCur=hk[P + p, :a], dCur=hd[P + p, :a], Tcw=T0[p], scale=sc, kLast=hk[p, :b], hasMP=np.ones(b, np.uint8), Xw=hX[p, :b], dLast=hd[p, :b],
                 mpObs=np.ones(b, np.int32), curTaken=np.zeros(a, np.uint8), faceW=650)
        c = _check_task(oracle, s, g, p, a, cth, T)
        assert c["count"] > 100, (p, c["count"])
        print("\nextracted task %d: %d / %d key points, %d matches, %d gathered, %d inliers" % (p, b, a, g["nm"][p], g["count"][p], g["inl"][p]))
