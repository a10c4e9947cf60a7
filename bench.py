#!/usr/bin/env python
"""bench.py — headline benchmark of the B200 hot path (BASELINE.json metric: "frames/sec ORB extract+match & LocalBA iters/sec").

  python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU under torchrun for N>1)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path on the host cores

Workload at N=1 = BASELINE.json configs[1] (+ the matching of configs[2] on the extracted descriptors): batched fisheye->cubemap warp + ORB
extraction of 4096 synthetic 1280x1024 frames, 650-px faces (front_cam_params.yaml with Ih=1024, nFeatures 3000), then the all-pairs 256-bit
Hamming matcher between every pair of consecutive frames. A "step" is one pass over all 4096 frames (launched in batches of --batch).
Frames are sharded over ranks without any collective; per-rank work is fixed ("weak" scaling), `value` is the whole-job frames/s =
N * frames * K / max-over-ranks device time. LocalBA LM iterations/s (configs[3], the second half of the metric), the 2000x2000 matcher
of configs[2], PoseOptimization and the config-5 tracking pipeline are separate legs under "extra", each with its own roofline / cpu_baseline / e2e.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from cubemapslam_b200 import config, synth  # noqa: E402

N_BASE = 16          # distinct synthetic frames generated with the SURVEY §8d recipe; the rest are circular shifts of them
METRIC = "warp+ORB-extract+match frames/sec"


def load_mask():
    return config.load_mask("gray_cubemap_front_mask_650")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clock / throttle-reason sampling during the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx = gpu_index; self.rows = []; self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True); self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = []; mx = None; reasons = set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = float(r[2])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def make_frames_device(torch, cfg, frames, device):
    """frames x Ih x Iw uint8 on the device: N_BASE recipe frames, the others are horizontal rolls re-masked by the image circle."""
    import math
    Iw, Ih = int(cfg["Camera.Iw"]), int(cfg["Camera.Ih"])
    base = np.stack([synth.fisheye_frame(cfg, i) for i in range(min(N_BASE, frames))])
    tb = torch.from_numpy(base).to(device)
    yy, xx = np.mgrid[0:Ih, 0:Iw]
    invp = [cfg.get("Camera.pol%d" % i, 0.0) for i in range(int(cfg["Camera.nrinvpol"]))]
    fov = cfg["Camera.fov"] / 2.0 * math.pi / 180.0
    rho = synth._horner(invp, math.atan(-math.cos(fov) / math.sin(fov)))
    circle = torch.from_numpy(((xx - cfg["Camera.u0"]) ** 2 + (yy - cfg["Camera.v0"]) ** 2 <= rho ** 2)).to(device)
    out = torch.empty((frames, Ih, Iw), dtype=torch.uint8, device=device)
    for i in range(frames):
        b = tb[i % len(base)]
        shift = (i // len(base)) * 7
        out[i] = torch.roll(b, shifts=shift, dims=1) * circle if shift else b
    return out, base


def geometry_bytes(cfg, nlevels=8, scale=1.2):
    """Algorithmic bytes per frame of each kernel (SURVEY.md §8d): every input byte read once, every output written once."""
    Iw, Ih, W = int(cfg["Camera.Iw"]), int(cfg["Camera.Ih"]), int(cfg["CubeFace.w"])
    sizes = []; s = np.float32(1.0)
    for l in range(nlevels):
        inv = np.float32(1.0) / s
        sizes.append(int(np.rint(np.float32(3 * W) * inv)) ** 2)
        s = np.float32(s * np.float32(scale))
    # pixels FAST scores per level: the detection area of the cell grid, (side - 2 * 16 - 6)^2 (src/ORBExtractor.cpp:763-803)
    scored = sum(max(int(round(sz ** 0.5)) - 38, 0) ** 2 for sz in sizes)
    return {"k_warp": Iw * Ih + 5 * W * W, "k_pyramid": sum(sizes[:-1]) + sum(sizes[1:]), "k_fast": sum(sizes), "levels_px": sizes, "fast_scored_px": scored}


DUMP_FRAMES = 32     # frames whose full results --dump-outputs writes (a fixed, seeded sample; counts are written for every frame)


def dump_outputs(out_dir, kps, desc, nout, match, nmatch):
    """What the last timed step returned to its caller, as .npy files for comparing two builds output for output: per frame the key point
    and match counts, and for a seeded sample of frames the key points (x, y, size, angle, response, octave, class_id), the 32 descriptor
    bytes and the match index of every key point in the next frame. Entries past a frame's count (and the match row of the last frame,
    which has no next frame) are not computed by the step and are written as 0 / -1."""
    frames, cap = kps.shape[0], kps.shape[1]
    n = nout.cpu().numpy().astype(np.int64)
    pick = np.sort(np.random.default_rng(0).choice(frames, min(DUMP_FRAMES, frames), replace=False))
    k = kps[pick].cpu().numpy()
    fields = np.concatenate([k[..., :20].copy().view(np.float32), k[..., 20:].copy().view(np.int32).astype(np.float32)], axis=-1)
    live = np.arange(cap)[None, :] < n[pick][:, None]
    has_next = (pick < frames - 1)[:, None]
    out = {"keypoint_count": n.astype(np.float64),
           "match_count": np.where(np.arange(frames) < frames - 1, nmatch.cpu().numpy(), 0).astype(np.float64),
           "sample_frames": pick.astype(np.float64),
           "keypoints": np.where(live[..., None], fields, 0).astype(np.float32),
           "descriptors": np.where(live[..., None], desc[pick].cpu().numpy(), 0).astype(np.float32),
           "matches": np.where(live & has_next, match[pick].cpu().numpy(), -1).astype(np.float32)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    import torch
    from cubemapslam_b200.frontend import FrontEnd
    from cubemapslam_b200.matcher import ORBMatcher
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        # NCCL writes its version banner (NCCL_DEBUG >= VERSION, set in this image) to stdout: send NCCL's log to stderr, stdout carries the one JSON line only
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    cfg = config.front_1024()
    mask = load_mask()
    B = args.batch
    fe = FrontEnd(cfg, mask, max_batch=B, device=local)
    kp_cap = fe.kp_cap
    mt = ORBMatcher(0.6, True, max_pairs=B + 1, max_features=kp_cap, device=local)
    frames = args.frames
    fish, base_host = make_frames_device(torch, cfg, frames, dev)
    fsz = fish.shape[1] * fish.shape[2]
    kps = torch.empty((frames, kp_cap, 28), dtype=torch.uint8, device=dev)
    desc = torch.empty((frames, kp_cap, 32), dtype=torch.uint8, device=dev)
    nout = torch.zeros((frames,), dtype=torch.int32, device=dev)
    match = torch.empty((frames, kp_cap), dtype=torch.int32, device=dev)
    nmatch = torch.zeros((frames,), dtype=torch.int32, device=dev)
    fs = torch.cuda.ExternalStream(fe.stream, device=dev); ms = torch.cuda.ExternalStream(mt.stream, device=dev)
    torch.cuda.synchronize()

    def one_step():
        fs.wait_stream(ms)                                          # the next pass overwrites buffers the matcher of the previous pass read
        for c in range(0, frames, B):
            b = min(B, frames - c)
            fe.run_dev(fish.data_ptr() + c * fsz, b, kps.data_ptr() + c * kp_cap * 28, desc.data_ptr() + c * kp_cap * 32, nout.data_ptr() + c * 4)
            ms.wait_stream(fs)
            f0 = max(c - 1, 0); nf = c + b - f0                     # pairs (f, f+1) whose second frame was just extracted
            if nf >= 2:
                mt.match_frames_dev(kps.data_ptr() + f0 * kp_cap * 28, desc.data_ptr() + f0 * kp_cap * 32, nout.data_ptr() + f0 * 4, kp_cap, nf,
                                    match.data_ptr() + f0 * kp_cap * 4, nmatch.data_ptr() + f0 * 4)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        one_step()
    fe.sync(); mt.sync()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = fe.launches + mt.launches
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(fs)
    for _ in range(args.steps):
        one_step()
    ms.wait_stream(fs)
    e1.record(ms)
    fe.sync(); mt.sync()
    barrier()
    ms_total = e0.elapsed_time(e1)
    launches = fe.launches + mt.launches - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, kps, desc, nout, match, nmatch)
    tms = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_max = float(tms.item())
    value = world * frames * args.steps / (ms_max / 1e3)
    nkp = float(nout.float().mean().item()); nmt = float(nmatch[:frames - 1].float().mean().item())

    # ---- end-to-end through the host entry points (pinned host frames in, host keypoints / descriptors / matches out)
    ef = min(args.e2e_frames, frames)
    h_in = torch.empty((ef, fish.shape[1], fish.shape[2]), dtype=torch.uint8).pin_memory()
    h_in.copy_(fish[:ef].cpu())
    KP = np.dtype([("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"), ("octave", "<i4"), ("class_id", "<i4")])
    # two sets of pinned result buffers: the matcher call of batch i (a worker thread; ctypes drops the GIL inside the C call) overlaps the front-end call
    # of batch i+1 - two synchronous host calls of the public API pipelined by the application, like the reference's own Tracking / LocalMapping threads
    from concurrent.futures import ThreadPoolExecutor
    sets = []
    for _ in range(2):
        t_kps = torch.empty((B + 1, kp_cap, 28), dtype=torch.uint8).pin_memory(); t_desc = torch.empty((B + 1, kp_cap, 32), dtype=torch.uint8).pin_memory()
        t_n = torch.empty((B + 1,), dtype=torch.int32).pin_memory()
        sets.append((t_kps, t_desc, t_n, t_kps.numpy(), t_desc.numpy(), t_n.numpy()))
    h_np = h_in.numpy()
    pool = ThreadPoolExecutor(max_workers=1)

    def match_job(k, lo, b):
        _, _, _, h_kps, h_desc, h_n = sets[k]
        nm_, _m = mt.match_frames(h_kps[lo:b + 1].view(KP).reshape(b + 1 - lo, kp_cap), h_desc[lo:b + 1], h_n[lo:b + 1])
        return int(nm_.sum())

    def e2e_pass():
        tot = 0; prev = None; pending = [None, None]; k = 0
        for c in range(0, ef, B):
            b = min(B, ef - c)
            if pending[k] is not None:
                tot += pending[k].result(); pending[k] = None      # this buffer set is free again
            _, _, _, h_kps, h_desc, h_n = sets[k]
            fe.run_raw(h_np[c:c + b], h_kps[1:], h_desc[1:], h_n[1:])
            lo = 1
            if prev is not None:   # slot 0 keeps the last frame of the previous batch so that every consecutive pair is matched
                pk, pb = prev
                h_kps[0] = sets[pk][3][pb]; h_desc[0] = sets[pk][4][pb]; h_n[0] = sets[pk][5][pb]; lo = 0
            pending[k] = pool.submit(match_job, k, lo, b)
            prev = (k, b); k ^= 1
        for f in pending:
            if f is not None:
                tot += f.result()
        return tot
    e2e_pass()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        e2e_pass()
    barrier()
    t_e2e = time.perf_counter() - t0
    te = torch.tensor([t_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * ef * args.e2e_steps / float(te.item())
    h2d = ef * fsz + ef * kp_cap * 60 + ef * 4               # frames in; key points + descriptors + counts re-uploaded by the host matcher call
    d2h = ef * (kp_cap * 60 + 4) + ef * (kp_cap * 4 + 4)     # key points, descriptors, counts; match indices, match counts

    sharded = None
    if world > 1 and not args.no_extra:
        import bench_extra
        sharded = bench_extra.run_multi(args, local, rank, world, dist, torch)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- per-kernel roofline (separate short pass with events between launches)
    gb = geometry_bytes(cfg)
    hbm, tf, how = peaks()
    fe.set_timing(True)
    nb = min(frames, 4 * B) // B
    me0 = torch.cuda.Event(enable_timing=True); me1 = torch.cuda.Event(enable_timing=True); mms = 0.0
    for c in range(0, nb * B, B):
        fe.run_dev(fish.data_ptr() + c * fsz, B, kps.data_ptr() + c * kp_cap * 28, desc.data_ptr() + c * kp_cap * 32, nout.data_ptr() + c * 4)
        fe.sync()
        me0.record(ms)
        mt.match_frames_dev(kps.data_ptr() + c * kp_cap * 28, desc.data_ptr() + c * kp_cap * 32, nout.data_ptr() + c * 4, kp_cap, B, match.data_ptr() + c * kp_cap * 4, nmatch.data_ptr() + c * 4)
        me1.record(ms); mt.sync()
        mms += me0.elapsed_time(me1)
    tm = fe.timing(); fe.set_timing(False)
    tm["k_match_bruteforce"] = (mms, nb)
    total_ms = sum(v[0] for v in tm.values()) or 1.0
    popc_peak = mt.ubench_popc()
    mm3_peak = mt.ubench_minmax3()
    algo = {"k_warp": gb["k_warp"], "k_pyramid": gb["k_pyramid"], "k_fast": gb["k_fast"], "k_describe": int(nkp * (43 * 43 + 31 * 31 + 60)), "k_distribute": None,
            "k_match_bruteforce": int(2 * nkp * 36 + nkp * 8)}
    traffic_tab = {}
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        traffic_tab = json.load(open(tp)).get("dram_bytes_per_frame", {})
    per_kernel = {}
    for k, (kms, _) in tm.items():
        ent = {"share_of_step": round(kms / total_ms, 4), "ms_per_batch": round(kms / nb, 4)}
        if algo.get(k):
            ent["algorithmic_bytes_per_frame"] = algo[k]
            ent["achieved_GBs"] = round(algo[k] * B / (kms / nb / 1e3) / 1e9, 2)
            ent["frac_of_hbm"] = round(ent["achieved_GBs"] / hbm, 4)
        if k == "k_match_bruteforce":
            popc = (B - 1) * nkp * nkp * 8 / (kms / nb / 1e3)
            ent.update({"bound": "popc issue", "achieved_popc32_per_s": round(popc, 3), "measured_peak_popc32_per_s": round(popc_peak, 3), "frac_of_popc_peak": round(popc / popc_peak, 4)})
        if k == "k_fast":   # exact arc score = 80 three-input u16x2 min/max per pixel pair (DESIGN.md §4): the instruction the kernel is bound by
            mm3 = 40.0 * gb["fast_scored_px"] * B / (kms / nb / 1e3)
            ent.update({"bound": "int ALU issue (VIMNMX3.U16x2)", "scored_px_per_frame": gb["fast_scored_px"], "achieved_minmax3_per_s": round(mm3, 1),
                        "measured_peak_minmax3_per_s": round(mm3_peak, 1), "frac_of_minmax3_peak": round(mm3 / mm3_peak, 4),
                        "peak_source": "cslam_ubench_minmax3 on this GPU (register-only VIMNMX3.U16x2 chains)"})
        per_kernel[k] = ent
    dom = max(tm, key=lambda k: tm[k][0])
    roof = {"kernel": dom, "bound": "hbm", "peak": hbm, "peak_source": how, "unit": "GB/s", "share_of_step": per_kernel[dom]["share_of_step"],
            "achieved": per_kernel[dom].get("achieved_GBs"), "frac": per_kernel[dom].get("frac_of_hbm"),
            "traffic": int(traffic_tab[dom] * B) if dom in traffic_tab else None, "per_kernel": per_kernel}
    if dom == "k_fast":
        roof["note"] = ("k_fast is integer-ALU bound, not HBM bound (ncu: ALU pipe ~68 % active, DRAM 2-3 %): `frac` is reported against HBM as the contract asks; "
                        "its real bound is per_kernel.k_fast.frac_of_minmax3_peak (score arithmetic alone against a measured VIMNMX3 peak); DESIGN.md §4")
    whole = sum(v for v in [gb["k_warp"], gb["k_pyramid"], gb["k_fast"], 2 * gb["k_fast"], int(nkp * (43 * 43 + 31 * 31)), algo["k_match_bruteforce"]])
    roof["pipeline_algorithmic_bytes_per_frame"] = whole          # SURVEY §8d accounting (incl. the reference's whole-level blur) + matcher I/O
    roof["pipeline_frac"] = round(whole * (value / world) / 1e9 / hbm, 4)

    cpu = cpu_baseline(cfg, mask, base_host, args)
    extra = {}
    if sharded is not None:
        extra = sharded
    elif not args.no_extra:
        import bench_extra
        fe.close(); mt.close()
        del fish, kps, desc, match
        torch.cuda.empty_cache()
        extra = bench_extra.run(args, local)
    out = {"metric": METRIC, "value": round(value, 1), "unit": "frames/s", "n_gpus": world, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": round(ms_max / args.steps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "u8", "data": "synthetic (SURVEY §8d recipe: %d distinct frames, others are re-masked circular shifts)" % N_BASE,
           "config": {"workload": "configs[1]+[2]: warp + ORB extract of %d synthetic 1280x1024 frames per GPU (650-px faces, nFeatures 3000) + all-pairs Hamming match of consecutive frames" % frames,
                      "frames_per_gpu": frames, "batch": B, "l2": "inputs (%.1f GB) larger than L2" % (frames * fsz / 1e9), "parallelism": "frame-shard x%d" % world,
                      "mean_keypoints_per_frame": round(nkp, 1), "mean_matches_per_pair": round(nmt, 1),
                      "second_metric": "LocalBA LM iterations/s: extra.local_ba.lm_iters_per_s"},
           "clocks": clocks, "gpu_launches": int(launches),
           "e2e": {"value": round(e2e_value, 1), "unit": "frames/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                   "frames_per_step": ef, "steps": args.e2e_steps, "calls": "cslam_frontend_run + cslam_match_frames (host buffers); the matcher call of batch i runs on a second host thread while the front-end call of batch i+1 runs"},
           "roofline": roof, "cpu_baseline": cpu, "extra": extra}
    emit(out)
    if world > 1:
        dist.destroy_process_group()


def host_cores():
    """CPUs this process may really use: the cgroup CPU quota if there is one (the GPU boxes expose 128 logical CPUs but a
    16-CPU quota), else os.cpu_count()."""
    n = os.cpu_count() or 1
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(round(int(q) / int(per)))))
    except Exception:
        pass
    return n


def cv2_primitive_ms(cfg):
    """opencv-python 4.13 wall time of the bare OpenCV primitives on one 1950^2 canvas, 1 thread: a sanity lower bound for any CPU path (SURVEY §8d)."""
    try:
        import cv2
    except Exception:
        return None
    cv2.setNumThreads(1)
    rng = np.random.default_rng(0)
    W3 = 3 * int(cfg["CubeFace.w"])
    img = cv2.resize(rng.integers(0, 256, (W3 // 8, W3 // 8), dtype=np.uint8), (W3, W3))
    out = {}
    t0 = time.perf_counter(); lv = [img]
    for l in range(1, 8):
        s = int(round(W3 / 1.2 ** l)); lv.append(cv2.resize(lv[-1], (s, s), interpolation=cv2.INTER_LINEAR))
    out["pyramid_ms"] = round(1e3 * (time.perf_counter() - t0), 2)
    t0 = time.perf_counter()
    for a in lv:
        cv2.GaussianBlur(a, (7, 7), 2, 2, borderType=cv2.BORDER_REFLECT_101)
    out["blur_ms"] = round(1e3 * (time.perf_counter() - t0), 2)
    fd = cv2.FastFeatureDetector_create(20, True, cv2.FAST_FEATURE_DETECTOR_TYPE_9_16)
    t0 = time.perf_counter()
    for a in lv:
        fd.detect(a)
    out["fast_whole_image_ms"] = round(1e3 * (time.perf_counter() - t0), 2)
    m = rng.uniform(0, 1000, (int(cfg["CubeFace.w"]), int(cfg["CubeFace.w"]))).astype(np.float32)
    src = rng.integers(0, 256, (int(cfg["Camera.Ih"]), int(cfg["Camera.Iw"])), dtype=np.uint8)
    t0 = time.perf_counter()
    for _ in range(5):
        cv2.remap(src, m, m, cv2.INTER_LINEAR)
    out["remap_5_faces_ms"] = round(1e3 * (time.perf_counter() - t0), 2)
    out["threads"] = 1
    return out


def cpu_baseline(cfg, mask, base_frames, args, threads=None, nframes=None, with_cv2=True):
    """Warp + extract + consecutive-frame matching on the host cores, bounded sample. Extraction runs the reference's OWN ORBExtractor.cpp /
    CamModelGeneral.cpp (oracle/_ref/libref.so, compiled unmodified against the cv:: shim) when that library travelled with the tree, else the
    oracle port; the all-pairs matcher has no reference function (DESIGN.md §2) and is the oracle port in both cases."""
    import oracle as orc
    quota = host_cores()
    cores = threads or min(os.cpu_count() or 1, 2 * quota)     # 2 worker threads per granted CPU measured fastest on the box
    cp = orc.cam_params(cfg)
    m1, m2 = orc.build_maps(cp)
    n = nframes or 16 * cores
    fr = np.stack([base_frames[i % len(base_frames)] for i in range(n)])
    cap = 3000 + 24
    kind = "port"
    try:
        from oracle import ref as R
        if R.available():
            kind = "reference"
    except Exception:
        pass
    if kind == "reference":
        r = R.Ref(cp)
        r.warp_extract_batch_out(fr[:min(n, cores)], m1, m2, mask, 3000, 1.2, 8, 20, 7, cores, cap)     # warm-up
        t0 = time.perf_counter()
        kps, desc, nn = r.warp_extract_batch_out(fr, m1, m2, mask, 3000, 1.2, 8, 20, 7, cores, cap)
        t_ext = time.perf_counter() - t0
        t0 = time.perf_counter()
        r.warp_extract_batch_out(fr[:max(4, n // 8)], m1, m2, mask, 3000, 1.2, 8, 20, 7, 1, cap)
        t_one = (time.perf_counter() - t0) / max(4, n // 8)
    else:
        orc.warp_extract_batch_out(cp, fr[:min(n, cores)], m1, m2, mask, 3000, 1.2, 8, 20, 7, cores, cap)
        t0 = time.perf_counter()
        kps, desc, nn = orc.warp_extract_batch_out(cp, fr, m1, m2, mask, 3000, 1.2, 8, 20, 7, cores, cap)
        t_ext = time.perf_counter() - t0
        t0 = time.perf_counter()
        orc.warp_extract_batch_out(cp, fr[:max(4, n // 8)], m1, m2, mask, 3000, 1.2, 8, 20, 7, 1, cap)
        t_one = (time.perf_counter() - t0) / max(4, n // 8)
    t0 = time.perf_counter()
    nm, _ = orc.match_frames_batch(kps, desc, nn, 0.6, 50, True, nthreads=cores)
    t_match = time.perf_counter() - t0
    dt = t_ext + t_match
    out = {"value": round(n / dt, 2), "unit": "frames/s", "cores": quota, "threads": cores, "kind": kind,
           "sample": "%d frames of the same workload, %d independent worker threads on %d granted CPUs; extraction = %s, matching = oracle port (-O3)"
                     % (n, cores, quota, "the reference's ORBExtractor.cpp compiled unmodified (oracle/_ref)" if kind == "reference" else "oracle port"),
           "seconds": round(dt, 2), "extract_frames_per_s": round(n / t_ext, 2), "match_pairs_per_s": round((n - 1) / max(t_match, 1e-9), 2),
           "single_thread_extract_frames_per_s": round(1.0 / t_one, 2), "mean_keypoints_per_frame": round(float(nn.mean()), 1), "mean_matches_per_pair": round(float(nm[:n - 1].mean()), 1)}
    if with_cv2:
        out["cv2_primitives_1_thread"] = cv2_primitive_ms(cfg)
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = config.front_1024()
    mask = load_mask()
    base = np.stack([synth.fisheye_frame(cfg, i) for i in range(N_BASE)])
    vals = []
    for i in range(args.warmup + args.steps):
        c = cpu_baseline(cfg, mask, base, args, nframes=192, with_cv2=(i == args.warmup + args.steps - 1))
        if i >= args.warmup:
            vals.append(c)
    v = float(np.mean([c["value"] for c in vals]))
    c = vals[-1]; c["value"] = round(v, 2)
    out = {"impl": "reference", "metric": METRIC, "value": round(v, 2), "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": round(1e3 * c["seconds"], 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
           "data": "synthetic", "config": {"workload": "configs[1]+[2]: warp + ORB extract + consecutive-frame match, 1280x1024 frames, 650-px faces, nFeatures 3000 (bounded sample of 192 frames per step)"},
           "cpu_baseline": c, "e2e": {"value": round(v, 2), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(out)


_RESULT_FD = None


def _claim_stdout():
    """stdout must carry exactly one JSON line. Libraries below us write there too (NCCL prints its version banner on stdout in this image,
    whatever NCCL_DEBUG_FILE says), so file descriptor 1 is pointed at stderr for the whole run and the result line goes to a private duplicate
    of the original stdout."""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(line.decode()); sys.stdout.flush()
    else:
        os.write(_RESULT_FD, line)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=4096)
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--e2e-frames", type=int, default=1024)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--match-pairs", type=int, default=4096)
    ap.add_argument("--match-steps", type=int, default=2)
    ap.add_argument("--pose-frames", type=int, default=2048)
    ap.add_argument("--track-frames", type=int, default=1024)
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
