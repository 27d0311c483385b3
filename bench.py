#!/usr/bin/env python3
"""bench.py — ORB extraction throughput of the B200 front-end (BASELINE.json metric) + matching extras.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" = one pass of the hot path (ORBextractor::operator(), reference ORBextractor.cc:1083-1169)
over one batch of B synthetic 640x480 frames per GPU (TUM settings: 1000 features, 8 levels, 1.2,
FAST 20/7 — BASELINE config 1).  Frames are sharded by rank with no data-path collective (weak
scaling; SURVEY §8e).  One JSON line is printed by rank 0:
  value      frames/s with the batch already resident in HBM (device pointers in, device results out)
  e2e        frames/s through the host-pointer C-ABI call (pinned host frames -> H2D -> kernels -> D2H)
  roofline   the dominant kernel group's algorithmic bytes / its CUDA-event time vs the measured HBM peak
  cpu_baseline  the reference's own ORBextractor.cc (oracle/_ref, compiled unmodified) on this box's host cores, bounded sample
`--impl reference` times that CPU build alone (all host threads) and prints the same line shape.
`--dump-outputs DIR` writes rank 0's results of the last timed step as .npy files (see dump_outputs), so that two builds
can be compared output for output: the frames are seeded, identical from run to run.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

W, H, NFEAT, NLEVELS, SCALE, INI_TH, MIN_TH = 640, 480, 1000, 8, 1.2, 20, 7
METRIC = "orb_extraction_frames_per_s_640x480_1000f"
UNIT = "frames/s"


DUMP_FRAMES = 64                   # frames whose keypoints and descriptors --dump-outputs writes (about 12 MB)


def dump_outputs(out_dir, kps_d, desc_d, n_d, mono_d):
    """What the device-resident path hands its caller for a batch, one float .npy per array:
      n.npy, mono.npy    (B,)  keypoint count and monoIndex of every frame of the batch
      frames.npy         (S,)  the sampled frames: a fixed seeded choice of S = min(B, DUMP_FRAMES)
      keypoints.npy      (S, M, 7) float64  x, y, size, angle, response, octave, class_id of the sampled frames
      descriptors.npy    (S, M, 32) float32 descriptor bytes of the sampled frames
    M is the largest keypoint count among the sampled frames; rows past a frame's own count are zero."""
    from visual_sgraphs_b200._lib import KEYPOINT_DTYPE
    import torch
    os.makedirs(out_dir, exist_ok=True)
    B = kps_d.shape[0]
    n, mono = n_d.cpu().numpy(), mono_d.cpu().numpy()
    frames = np.sort(np.random.default_rng(0).choice(B, min(B, DUMP_FRAMES), replace=False))
    m = int(n[frames].max()) if len(frames) else 0
    sel = torch.as_tensor(frames, device=kps_d.device)
    kps = np.ascontiguousarray(kps_d[sel, :m].cpu().numpy()).view(KEYPOINT_DTYPE).reshape(len(frames), m)
    desc = desc_d[sel, :m].cpu().numpy().astype(np.float32)
    keys = np.stack([kps[f].astype(np.float64) for f in KEYPOINT_DTYPE.names], axis=-1)
    valid = np.arange(m)[None, :] < n[frames][:, None]
    keys[~valid], desc[~valid] = 0, 0
    for name, a in (("n", n.astype(np.float64)), ("mono", mono.astype(np.float64)), ("frames", frames.astype(np.float64)),
                    ("keypoints", keys), ("descriptors", desc)):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def level_sizes(w, h):
    inv, s = [], np.float32(1.0)
    for _ in range(NLEVELS):
        inv.append(np.float32(1.0) / s)
        s = np.float32(float(s) * float(np.float32(SCALE)))
    return [(int(np.rint(np.float32(w) * i)), int(np.rint(np.float32(h) * i))) for i in inv]


def algorithmic_bytes(w, h, n_kp, fused):
    """SURVEY §8(d): per-stage compulsory bytes per frame. P = sum of level pixels.  With the fused FAST + blur grid
    (the default) the "fast" stage is that one kernel: it reads every level for FAST (P) and reads + writes every level
    for the blur (2P); the "blur" stage is then empty."""
    px = [a * b for a, b in level_sizes(w, h)]
    P, p0, p7 = sum(px), px[0], px[-1]
    stages = {
        "pyramid": (P - p7) + (P - p0),   # read L0..L6, write L1..L7
        "fast": 3 * P if fused else P,    # read every level once (+ blur: read + write every level)
        "blur": 0 if fused else 2 * P,
        "describe": 60 * n_kp,            # 28 B keypoint + 32 B descriptor per keypoint
        "octree": 0,                      # latency-bound bookkeeping; no roofline claim
    }
    return stages, 5 * P - p0 - p7 + 60 * n_kp


def make_frames(n, seed0):
    """n distinct corner-rich frames: 32 seeded synthetic frames (SURVEY §8d), each reused with circular shifts."""
    from visual_sgraphs_b200.synth import synth_frame
    base = [synth_frame(seed0 + i, W, H) for i in range(min(n, 32))]
    out = np.empty((n, H, W), np.uint8)
    for i in range(n):
        k = i // len(base)
        out[i] = np.roll(base[i % len(base)], (7 * k, 13 * k), (0, 1))
    return out


def ncu_pipes(kernel):
    """Issue-slot / ALU-pipe / tensor-pipe utilisation of the kernel from the same committed capture (what bounds a kernel
    that the byte roofline does not explain)."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return None
    d = json.load(open(p)).get(kernel, {})
    out = {k: d[k] for k in ("issue_active_pct", "alu_pipe_active_pct", "tensor_pipe_active_pct") if k in d}
    return out or None


def ncu_traffic(kernel, frames):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch from the committed ncu --set full capture
    (profiles/ncu_traffic.json), scaled from the captured frames per launch to this run's."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return None
    d = json.load(open(p))
    if kernel not in d:
        return None
    return d[kernel]["dram_bytes_per_launch"] / d["frames_per_launch"] * frames


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            self.nv = None

    def run(self):
        while not self.stop_flag and self.nv is not None:
            try:
                self.sm.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.004)

    def result(self):
        self.stop_flag = True
        if self.nv is None or not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml_unavailable"]}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.sm)}


def workload_config(B):
    """The `config` object — identical in the repo arm and the reference arm (the driver compares them)."""
    return {"workload": "C1: ORBextractor 640x480, 1000 features, 8 levels, scale 1.2, FAST 20/7",
            "frames_per_step_per_gpu": B, "sharding": "frames by rank, no collective",
            "l2": "inputs larger than L2: %d MB of frames + %d MB of pyramid/blur planes per step" %
                  (B * W * H >> 20, (2 * B * 1158012) >> 20)}


def cpu_reference():
    """(kind, bench_extract(frames, threads) -> (seconds, keypoints)).  kind "reference" = oracle/_ref/libvsg_ref.so, the
    reference's own ORBextractor.cc compiled unmodified (oracle/ref_build/Makefile); "port" = the oracle restatement,
    only when that library is neither prebuilt nor buildable."""
    try:
        from oracle import ref
        if ref.available():
            ref.lib()
            return "reference", lambda frames, threads: ref.bench_extract(frames, NFEAT, SCALE, NLEVELS, INI_TH, MIN_TH, threads)
    except Exception as e:  # noqa: BLE001
        print("oracle/_ref unavailable (%s); timing the oracle port instead" % e, file=sys.stderr)
    from oracle import oracle as orc
    return "port", lambda frames, threads: orc.bench_extract(frames, NFEAT, SCALE, NLEVELS, INI_TH, MIN_TH, threads)


def cpu_throughput(nframes, threads):
    """The reference's CPU extractor over `nframes` frames of the workload on `threads` host threads."""
    kind, fn = cpu_reference()
    frames = make_frames(nframes, 9000)
    fn(frames[:min(nframes, 4 * threads)], threads)          # untimed: first-touch of the per-thread malloc arenas
    secs, total_kp = fn(frames, threads)
    return kind, nframes / secs, secs, total_kp


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation of the path (oracle/_ref: ORBextractor.cc compiled
    unmodified; the oracle port only if that library is missing), all host threads (one extractor instance per thread,
    as Frame.cc:129-132 runs left / right), each step a bounded sample of the workload."""
    if rank != 0:
        return
    cores = host_threads()
    per_step = max(cores * 16, 64)
    kind, fn = cpu_reference()
    frames = make_frames(per_step, 9000)
    for _ in range(args.warmup):
        fn(frames[:cores], cores)
    secs = 0.0
    for _ in range(args.steps):
        s, _ = fn(frames, cores)
        secs += s
    value = per_step * args.steps / secs
    sample = "%d frames per step x %d steps, %d threads, one extractor per thread" % (per_step, args.steps, cores)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args.batch),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def latency_extras(torch, lib, device):
    """One frame per call through vsg_extract (the reference's per-frame operator() use): pinned frame in, pinned
    keypoints/descriptors out, host clock around each call."""
    from visual_sgraphs_b200._lib import check, ptr
    from visual_sgraphs_b200.extractor import ORBextractor
    import ctypes as C
    ex = ORBextractor(NFEAT, SCALE, NLEVELS, INI_TH, MIN_TH, device=device, max_batch=1)
    cap = ex.max_keypoints(W, H)
    frames = torch.from_numpy(make_frames(8, 4000)).pin_memory()
    kp = torch.zeros((cap, 28), dtype=torch.uint8).pin_memory()
    de = torch.zeros((cap, 32), dtype=torch.uint8).pin_memory()
    n, mono = C.c_int(0), C.c_int(0)
    fn = frames.numpy()

    def one(i):
        check(lib.vsg_extract(ex._h, ptr(fn[i % 8]), W, H, W, 0, 0, ptr(kp), ptr(de), cap, C.byref(n), C.byref(mono)))

    for i in range(20):
        one(i)
    ts = []
    for i in range(200):
        t0 = time.perf_counter()
        one(i)
        ts.append(time.perf_counter() - t0)
    ex.close()
    ts = np.array(ts) * 1e3
    return {"ms_median": float(np.median(ts)), "ms_p95": float(np.percentile(ts, 95)),
            "frames_per_s": float(1e3 / np.mean(ts)), "calls": 200}


def other_config_extras(torch, lib, device):
    """The other BASELINE configs as reported extras (they are parity-test cases, not bench lines): C4 1280x720 / 2000
    features (device-resident batch), C2 EuRoC-shaped stereo pairs through the host API (extraction of both images in
    one batched call + vsg_stereo_match on the device pyramids), C3 SearchByProjection of a 200k-point map into a
    1000-keypoint frame (one call, host arrays in and out)."""
    from visual_sgraphs_b200._lib import KEYPOINT_DTYPE, TRACK_POINT_DTYPE
    from visual_sgraphs_b200.extractor import ORBextractor
    from visual_sgraphs_b200.frame import FrameData
    from visual_sgraphs_b200.matcher import ORBmatcher
    from visual_sgraphs_b200.synth import synth_frame, synth_stereo_pair
    out = {}
    # ---- C4 ----
    B4 = 128
    base = [synth_frame(6000 + i, 1280, 720) for i in range(8)]
    fr = np.stack([np.roll(base[i % 8], (5 * (i // 8), 11 * (i // 8)), (0, 1)) for i in range(B4)])
    d_frames = torch.from_numpy(fr).cuda()
    ex = ORBextractor(2000, SCALE, NLEVELS, INI_TH, MIN_TH, device=device, max_batch=B4)
    cap = ex.max_keypoints(1280, 720)
    kps = torch.zeros((B4, cap, 28), dtype=torch.uint8, device="cuda")
    desc = torch.zeros((B4, cap, 32), dtype=torch.uint8, device="cuda")
    n = torch.zeros(B4, dtype=torch.int32, device="cuda")
    mono = torch.zeros(B4, dtype=torch.int32, device="cuda")
    st = torch.cuda.ExternalStream(ex.stream(), device=device)
    torch.cuda.synchronize()
    for _ in range(2):
        ex.extract_batch_dev(d_frames, kps, desc, n, mono)
    ex.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(5):
        ex.extract_batch_dev(d_frames, kps, desc, n, mono)
    e1.record(st)
    ex.sync()
    ms = e0.elapsed_time(e1) / 5
    out["c4_1280x720_2000f"] = {"frames_per_s": B4 / (ms * 1e-3), "ms_per_128_frames": ms,
                                "keypoints_per_frame": float(n.float().mean().item())}
    # beside it: the reference's CPU extractor on the same shape (all host threads), and the pipeline's algorithmic bytes
    # (SURVEY 8d: B_frame = 5P - p0 - p7 + 60N) against the measured HBM peak
    cores = host_threads()
    try:
        from oracle import ref
        kind = "reference"
        secs, _ = ref.bench_extract(fr[: 4 * cores], 2000, SCALE, NLEVELS, INI_TH, MIN_TH, cores)
    except Exception:  # noqa: BLE001
        from oracle import oracle as orc
        kind = "port"
        secs, _ = orc.bench_extract(fr[: 4 * cores], 2000, SCALE, NLEVELS, INI_TH, MIN_TH, cores)
    px = [a * b for a, b in level_sizes(1280, 720)]
    b_frame = 5 * sum(px) - px[0] - px[-1] + 60 * float(n.float().mean().item())
    peak, peak_src = measured_peaks()
    out["c4_1280x720_2000f"]["cpu_baseline"] = {"value": 4 * cores / secs, "unit": "frames/s", "cores": cores, "kind": kind,
                                                "sample": "%d frames, %d threads" % (4 * cores, cores)}
    out["c4_1280x720_2000f"]["roofline"] = {"bound": "hbm", "achieved": b_frame * B4 / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                            "frac": b_frame * B4 / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_frame": b_frame,
                                            "scope": "whole pipeline (all kernels of the batch)", "peak_source": peak_src}
    ex.close()
    del d_frames, kps, desc
    # ---- C2 ----
    npairs = 64
    base_pairs = [synth_stereo_pair(8000 + i) for i in range(8)]
    pairs = [base_pairs[i % 8] for i in range(npairs)]
    stack = torch.from_numpy(np.stack([im for pr in pairs for im in pr])).pin_memory()   # L0 R0 L1 R1 ...
    ex2 = ORBextractor(1200, SCALE, NLEVELS, INI_TH, MIN_TH, device=device, max_batch=2 * npairs)
    m = ORBmatcher(device=device)

    from visual_sgraphs_b200._lib import check, ptr
    cap2 = ex2.max_keypoints(752, 480)
    kp2 = torch.zeros((2 * npairs, cap2, 28), dtype=torch.uint8).pin_memory()
    de2 = torch.zeros((2 * npairs, cap2, 32), dtype=torch.uint8).pin_memory()
    n2, mono2 = np.zeros(2 * npairs, np.int32), np.zeros(2 * npairs, np.int32)
    u2 = torch.zeros((npairs, cap2), dtype=torch.float32).pin_memory()
    d2 = torch.zeros((npairs, cap2), dtype=torch.float32).pin_memory()
    stack_np = stack.numpy()

    def stereo_step():
        check(lib.vsg_extract_batch(ex2._h, ptr(stack_np), 2 * npairs, 752, 480, 752, 752 * 480, 0, 0, ptr(kp2), ptr(de2), cap2,
                                    ptr(n2), ptr(mono2)))
        check(lib.vsg_stereo_match_batch(m._h, ex2._h, npairs, 0.11, 47.9, ptr(u2), ptr(d2), cap2))   # pairs (2p, 2p+1)
        return int((u2 >= 0).sum())

    stereo_step()
    t0 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        matched = stereo_step()
    dt = (time.perf_counter() - t0) / reps
    out["c2_stereo_752x480_1200f"] = {"pairs_per_s": npairs / dt, "ms_per_pair": 1e3 * dt / npairs, "pairs_per_call": npairs,
                                      "stereo_matches_per_pair": matched / npairs,
                                      "api": "vsg_extract_batch (pinned frames in) + vsg_stereo_match_batch (u_right / depth out)"}
    # beside it: the reference's path on the CPU for a sample of the same pairs — left / right extraction on two threads
    # (Frame.cc:129-132, oracle/_ref when present) + ComputeStereoMatches (oracle port), pairs dealt over the host threads
    try:
        import concurrent.futures as cf
        from oracle import oracle as orc
        def one_pair(pr):
            exl, exr = orc.OracleExtractor(1200), orc.OracleExtractor(1200)
            with cf.ThreadPoolExecutor(2) as tp:
                (ml, kl, dl), (mr, kr, dr) = tp.map(lambda a: a[0](a[1]), ((exl, pr[0]), (exr, pr[1])))
            return orc.stereo_matches(exl, exr, kl, dl, kr, dr, 0.11, 47.9)
        cores = host_threads()
        sample = [base_pairs[i % 8] for i in range(max(8, cores))]
        one_pair(sample[0])
        t0 = time.perf_counter()
        with cf.ThreadPoolExecutor(max(1, cores // 2)) as tp:
            list(tp.map(one_pair, sample))
        dt_cpu = time.perf_counter() - t0
        out["c2_stereo_752x480_1200f"]["cpu_baseline"] = {"value": len(sample) / dt_cpu, "unit": "pairs/s", "cores": cores, "kind": "port",
                                                          "sample": "%d pairs, %d workers x 2 extraction threads (ctypes calls release the GIL)" %
                                                                    (len(sample), max(1, cores // 2))}
    except Exception as e:  # noqa: BLE001
        out["c2_stereo_752x480_1200f"]["cpu_baseline"] = {"error": str(e)}
    # the same with the rectification System::TrackStereo runs first (System.cc:284-292; EuRoC.yaml needs it): unrectified
    # frames in, cv::remap on the device with one map per camera, then extraction + stereo matching
    ys, xs = np.meshgrid(np.arange(480, dtype=np.float64), np.arange(752, dtype=np.float64), indexing="ij")
    for slot, (k1, shift) in enumerate(((-0.05, 1.5), (-0.045, -1.0))):
        xn, yn = (xs - 376) / 450.0, (ys - 240) / 450.0
        f = 1 + k1 * (xn * xn + yn * yn)
        ex2.set_rectify_map(slot, (xn * f * 450 + 376 + shift).astype(np.float32), (yn * f * 450 + 240 - shift).astype(np.float32))

    def rectified_step():
        check(lib.vsg_extract_batch_rectify(ex2._h, ptr(stack_np), 2 * npairs, 752, 480, 752, 752 * 480, 2, 0, 0, ptr(kp2), ptr(de2),
                                            cap2, ptr(n2), ptr(mono2)))
        check(lib.vsg_stereo_match_batch(m._h, ex2._h, npairs, 0.11, 47.9, ptr(u2), ptr(d2), cap2))
        return int((u2 >= 0).sum())

    rectified_step()
    t0 = time.perf_counter()
    for _ in range(reps):
        matched_r = rectified_step()
    dtr = (time.perf_counter() - t0) / reps
    out["c2_stereo_752x480_1200f"]["rectified_on_device"] = {"pairs_per_s": npairs / dtr, "ms_per_pair": 1e3 * dtr / npairs,
                                                              "stereo_matches_per_pair": matched_r / npairs,
                                                              "api": "vsg_extract_batch_rectify (cv::remap per camera) + vsg_stereo_match_batch"}
    ex2.close()
    # ---- C3 ----
    rng = np.random.default_rng(3)
    n_kp, n_map = 1000, 200_000
    keys = np.zeros(n_kp, KEYPOINT_DTYPE)
    keys["x"], keys["y"] = rng.uniform(20, 620, n_kp), rng.uniform(20, 460, n_kp)
    keys["octave"] = rng.integers(0, 8, n_kp)
    kdesc = rng.integers(0, 256, (n_kp, 32), dtype=np.uint8)
    fdata = FrameData(keys, kdesc)
    src = rng.integers(0, n_kp, n_map)
    pts = np.zeros(n_map, TRACK_POINT_DTYPE)
    pts["proj_x"] = keys["x"][src] + rng.normal(0, 2, n_map)
    pts["proj_y"] = keys["y"][src] + rng.normal(0, 2, n_map)
    pts["view_cos"] = rng.uniform(0.99, 1.0, n_map)
    pts["level"] = np.clip(keys["octave"][src] + rng.integers(0, 2, n_map), 0, 7)
    pts["in_view"], pts["blocks"] = True, rng.random(n_map) < 0.9
    mp_desc = kdesc[src] ^ np.packbits(rng.random((n_map, 32, 8)) < 0.08, axis=2).reshape(n_map, 32)
    occ = np.zeros(n_kp, np.uint8)
    frame = m.frame(fdata)
    m.SearchByProjectionMap(frame, occ, pts, mp_desc, 3.0)
    t0 = time.perf_counter()
    for _ in range(5):
        nm, _ = m.SearchByProjectionMap(frame, occ, pts, mp_desc, 3.0)
    dt = (time.perf_counter() - t0) / 5
    out["c3_projection_1000kp_x_200k_map"] = {"ms_per_call": dt * 1e3, "map_points_per_s": n_map / dt, "nmatches": nm}
    try:   # beside it: the oracle port of ORBmatcher.cc:42-144 on the same scenario, one host thread (as Tracking calls it)
        from oracle import oracle as orc
        t0 = time.perf_counter()
        wnm, wassign = orc.search_by_projection_map(fdata.view, occ, pts, mp_desc, 3.0, False, 50.0, float(m.mfNNratio))
        dt_cpu = time.perf_counter() - t0
        _, assign_g = m.SearchByProjectionMap(frame, occ, pts, mp_desc, 3.0)
        out["c3_projection_1000kp_x_200k_map"]["cpu_baseline"] = {"value": dt_cpu * 1e3, "unit": "ms per call", "cores": 1, "kind": "port",
                                                                  "identical_results": bool(wnm == nm and np.array_equal(wassign, assign_g))}
    except Exception as e:  # noqa: BLE001
        out["c3_projection_1000kp_x_200k_map"]["cpu_baseline"] = {"error": str(e)}
    m.close()
    return out


def measured_popc_peak():
    """POPC results per second of this GPU, measured now by tools/micro/popc_peak (built by __graft_entry__.build());
    falls back to 16 / clk / SM at the measured SM clock (CUDA programming guide) if the binary is missing."""
    exe = os.path.join(ROOT, "tools", "micro", "popc_peak")
    try:
        import subprocess
        out = subprocess.run([exe], capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[-1]
        d = json.loads(out)
        return float(d["popc_per_s"]), "measured in this run (tools/micro/popc_peak: %.2f POPC / clk / SM)" % d["popc_per_clk_per_sm"]
    except Exception:  # noqa: BLE001
        return 16.0 * 148 * 1965e6, "fallback: 16 POPC / clk / SM x 148 SMs x 1965 MHz"


def measured_int8_peak():
    """Dense int8 tensor peak in OP/s: twice the measured dense bf16 rate of MEASURED_PEAKS.json (the tensor cores run 8-bit
    operands at twice the 16-bit rate; the file has no int8 entry), else the nominal 4.5e15."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        if "bf16_tflops" in d:
            return 2.0 * float(d["bf16_tflops"]) * 1e12, "2 x measured dense bf16 (MEASURED_PEAKS.json: %.0f TFLOP/s)" % d["bf16_tflops"]
    return 4.5e15, "nominal dense int8 (B200_PROFILING.md)"


def matching_extras(torch, device):
    """Hamming matching throughput (BASELINE metric part 2): brute-force kNN-2, configs C5 (100k x 1M) and C3's shape
    (1000 x 200k), device-resident descriptors, CUDA events on the matcher stream.  Two kernels, identical results: the
    tensor-core formulation (csrc/knn_tc.cu: tcgen05.mma.kind::i8 on +-1 expanded descriptors; the default for large
    problems) against the int8 tensor roofline, and the POPC kernel (VSG_KNN_TC=0) against the measured POPC peak."""
    from visual_sgraphs_b200.matcher import ORBmatcher
    m = ORBmatcher(device=device)
    s = torch.cuda.ExternalStream(m.stream(), device=device)
    out = {}
    g = torch.Generator(device="cuda").manual_seed(7)
    popc_peak, popc_src = measured_popc_peak()
    int8_peak, int8_src = measured_int8_peak()
    for name, nq, nt, reps in (("knn2_100k_x_1M", 100_000, 1_000_000, 3), ("knn2_1000_x_200k", 1000, 200_000, 20)):
        q = torch.randint(0, 256, (nq, 32), dtype=torch.uint8, device="cuda", generator=g)
        t = torch.randint(0, 256, (nt, 32), dtype=torch.uint8, device="cuda", generator=g)
        pairs = nq * nt
        res = {}
        for mode, label in (("2", "tensor"), ("0", "popc")):
            os.environ["VSG_KNN_TC"] = mode
            idx = torch.zeros((nq, 2), dtype=torch.int32, device="cuda")
            dist = torch.zeros((nq, 2), dtype=torch.int32, device="cuda")
            torch.cuda.synchronize()
            m.knn2_dev(q, t, idx, dist)
            m.sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(s)
            for _ in range(reps):
                m.knn2_dev(q, t, idx, dist)
            e1.record(s)
            m.sync()
            res[label] = (e0.elapsed_time(e1) / reps, idx, dist)
        os.environ.pop("VSG_KNN_TC", None)
        assert torch.equal(res["tensor"][1], res["popc"][1]) and torch.equal(res["tensor"][2], res["popc"][2])
        ms, ms_p = res["tensor"][0], res["popc"][0]
        ops = 2.0 * 256 * pairs / (ms * 1e-3)                 # s8 multiply-adds counted as 2 ops, K = 256
        out[name] = {"ms": ms, "pairs_per_s": pairs / (ms * 1e-3), "matches_per_s": nq / (ms * 1e-3),
                     "kernel": "knn2_tc_kernel (tcgen05.mma.kind::i8, TMA, TMEM epilogue)",
                     "roofline": {"bound": "tensor", "achieved": ops / 1e12, "peak": int8_peak / 1e12, "unit": "TOP/s (int8)",
                                  "frac": ops / int8_peak, "peak_source": int8_src, "frac_of_nominal_4500": ops / 4.5e15},
                     "popc_kernel": {"ms": ms_p, "pairs_per_s": pairs / (ms_p * 1e-3), "identical_results": True,
                                     "roofline": {"bound": "popc (xu pipe)", "achieved": 8 * pairs / (ms_p * 1e-3), "peak": popc_peak,
                                                  "unit": "POPC/s", "frac": 8 * pairs / (ms_p * 1e-3) / popc_peak,
                                                  "peak_source": popc_src}},
                     "speedup_over_popc_kernel": ms_p / ms}
    # CPU baseline beside it (SURVEY 8d): the reference's brute-force loop with its bit-hack DescriptorDistance
    # (ORBmatcher.cc:2047-2063) and a __builtin_popcountll variant, built with the reference's flags (-O3, no -march),
    # all host threads, bounded sample; the GPU result on the same sample must be identical
    from oracle import oracle as orc
    cores = host_threads()
    nq, nt = 512, 200_000
    q = torch.randint(0, 256, (nq, 32), dtype=torch.uint8, device="cuda", generator=g)
    t = torch.randint(0, 256, (nt, 32), dtype=torch.uint8, device="cuda", generator=g)
    idx = torch.zeros((nq, 2), dtype=torch.int32, device="cuda")
    dist = torch.zeros((nq, 2), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    m.knn2_dev(q, t, idx, dist)
    m.sync()
    qh, th = q.cpu().numpy(), t.cpu().numpy()
    cpu = {}
    for variant, label in ((0, "bit_hack"), (1, "popcountll")):
        secs, ci, cd = orc.bench_knn2(qh, th, cores, variant)
        assert np.array_equal(ci, idx.cpu().numpy()) and np.array_equal(cd, dist.cpu().numpy())
        cpu[label + "_pairs_per_s"] = nq * nt / secs
    cpu.update({"cores": cores, "kind": "port", "sample": "%d x %d descriptors, %d threads" % (nq, nt, cores)})
    out["cpu_baseline"] = cpu
    m.close()
    return out


def sharded_matching_extras(torch, dist, local_rank, rank, world):
    """The two matcher paths with a real exchange step, through the C ABI's communicator (vsg_comm_*: NCCL behind
    include/vsg_cuda.h, no Python on the data path): C5 brute-force kNN-2 with the 1M train descriptors sharded over the
    ranks (vsg_knn2_sharded: local search, ncclAllGather of the top-2 lists, (dist, idx) merge) and C3
    SearchByProjection of a 200k-point map sharded over the ranks into a 1000-keypoint frame
    (vsg_search_by_projection_map_sharded: claim-state token + ncclAllGather of the assignments).  Every rank's result is
    compared with the single-GPU call on the whole set.  Runs on every rank (collective); rank 0 returns the numbers."""
    from visual_sgraphs_b200._lib import KEYPOINT_DTYPE, TRACK_POINT_DTYPE
    from visual_sgraphs_b200.comm import Comm
    from visual_sgraphs_b200.frame import FrameData
    from visual_sgraphs_b200.matcher import ORBmatcher
    from visual_sgraphs_b200.sharded import shard_bounds
    comm = Comm.from_torch_distributed(dist, local_rank) if world > 1 else Comm(Comm.unique_id(), 1, 0, local_rank)
    m = ORBmatcher(nnratio=0.8, device=local_rank)
    s = torch.cuda.ExternalStream(m.stream(), device=local_rank)
    out = {"nccl_version": Comm.nccl_version(), "ranks": world}

    def sync_all():
        m.sync()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- C5: 100k x 1M, train rows sharded ----
    nq, nt = 100_000, 1_000_000
    g = torch.Generator(device="cuda").manual_seed(7)                 # same seed on every rank: same descriptors
    q = torch.randint(0, 256, (nq, 32), dtype=torch.uint8, device="cuda", generator=g)
    t = torch.randint(0, 256, (nt, 32), dtype=torch.uint8, device="cuda", generator=g)
    b, e = shard_bounds(nt, world)[rank]
    shard = t[b:e].contiguous()
    idx = torch.zeros((nq, 2), dtype=torch.int32, device="cuda")
    dd = torch.zeros((nq, 2), dtype=torch.int32, device="cuda")
    m.knn2_sharded(comm, q, shard, b, idx, dd)
    sync_all()
    reps = 3
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    for _ in range(reps):
        m.knn2_sharded(comm, q, shard, b, idx, dd)
    e1.record(s)
    sync_all()
    ms = torch.tensor([e0.elapsed_time(e1) / reps], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ref_i = torch.zeros_like(idx)
    ref_d = torch.zeros_like(dd)
    m.knn2_dev(q, t, ref_i, ref_d)                                    # the single-GPU call on the whole train set
    m.sync()
    same = bool(torch.equal(ref_i, idx) and torch.equal(ref_d, dd))
    assert same, "vsg_knn2_sharded differs from vsg_knn2_dev on rank %d" % rank
    out["c5_knn2_100k_x_1M_train_sharded"] = {"ms": float(ms[0]), "pairs_per_s": nq * nt / (float(ms[0]) * 1e-3),
                                              "matches_per_s": nq / (float(ms[0]) * 1e-3), "identical_to_single_gpu": same,
                                              "exchange": "ncclAllGather of %d B per rank" % (nq * 16)}
    del q, t, shard, idx, dd, ref_i, ref_d
    # ---- C3: 1000 keypoints x 200k map points, map sharded ----
    rng = np.random.default_rng(3)
    n_kp, n_map = 1000, 200_000
    keys = np.zeros(n_kp, KEYPOINT_DTYPE)
    keys["x"], keys["y"] = rng.uniform(20, 620, n_kp), rng.uniform(20, 460, n_kp)
    keys["octave"] = rng.integers(0, 8, n_kp)
    kdesc = rng.integers(0, 256, (n_kp, 32), dtype=np.uint8)
    fdata = FrameData(keys, kdesc)
    src = rng.integers(0, n_kp, n_map)
    pts = np.zeros(n_map, TRACK_POINT_DTYPE)
    pts["proj_x"] = keys["x"][src] + rng.normal(0, 2, n_map)
    pts["proj_y"] = keys["y"][src] + rng.normal(0, 2, n_map)
    pts["view_cos"] = rng.uniform(0.99, 1.0, n_map)
    pts["level"] = np.clip(keys["octave"][src] + rng.integers(0, 2, n_map), 0, 7)
    pts["in_view"], pts["blocks"] = True, rng.random(n_map) < 0.9
    mp_desc = kdesc[src] ^ np.packbits(rng.random((n_map, 32, 8)) < 0.08, axis=2).reshape(n_map, 32)
    occ = np.zeros(n_kp, np.uint8)
    frame = m.frame(fdata)
    b, e = shard_bounds(n_map, world)[rank]
    pts_l, desc_l = pts[b:e].copy(), mp_desc[b:e].copy()
    nm, assign = m.SearchByProjectionMapSharded(comm, frame, occ, b, pts_l, desc_l, 3.0)
    sync_all()
    reps = 5
    t0 = time.perf_counter()
    for _ in range(reps):
        nm, assign = m.SearchByProjectionMapSharded(comm, frame, occ, b, pts_l, desc_l, 3.0)
    sync_all()
    dt = torch.tensor([(time.perf_counter() - t0) / reps], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    m.SearchByProjectionMap(frame, occ, pts, mp_desc, 3.0)
    t0 = time.perf_counter()
    for _ in range(reps):
        nm1, assign1 = m.SearchByProjectionMap(frame, occ, pts, mp_desc, 3.0)
    dt1 = (time.perf_counter() - t0) / reps
    same = bool(nm == nm1 and np.array_equal(assign, assign1))
    assert same, "vsg_search_by_projection_map_sharded differs from the one-call method on rank %d" % rank
    out["c3_projection_1000kp_x_200k_map_sharded"] = {"ms_per_call": float(dt[0]) * 1e3, "map_points_per_s": n_map / float(dt[0]),
                                                      "single_gpu_ms_per_call": dt1 * 1e3, "nmatches": int(nm),
                                                      "identical_to_single_gpu": same,
                                                      "exchange": "%d-byte claim token down the ranks + ncclAllGather of %d B per rank" %
                                                                  (n_kp, 4 * (n_kp + 1))}
    m.close()
    comm.close()
    return out


_JSON_OUT = None


def reserve_stdout_for_the_json_line():
    """stdout carries exactly ONE line, the JSON result.  Anything libraries print there (NCCL prints its version line to
    stdout) is sent to stderr instead: fd 1 is pointed at fd 2 for the whole run and the JSON line goes to the saved fd."""
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def matching_methods_extras(device):
    """Every ORBmatcher method at tracking size (two related 640x480 frames, ~1000 features each): microseconds per call
    through the C ABI (host arrays in and out, the searched frame uploaded inside the timed call, as the drop-in shim does)
    beside the CPU oracle port of the same reference loop on the same scenario (one host thread, as the reference runs it).
    Results are asserted identical.  Scenario builders: tests/match_scenarios.py."""
    from oracle import oracle as orc
    from tests import match_scenarios as sc
    from visual_sgraphs_b200.matcher import ORBmatcher
    ka, da, kb, db = sc.two_frames(orc)
    rng = np.random.default_rng(5)
    out = {"features": [int(len(ka)), int(len(kb))], "unit": "us per call (median of 30)", "cpu_kind": "port, 1 thread"}

    def timed(fn, reps=30):
        fn()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            r = fn()
            ts.append(time.perf_counter() - t0)
        return float(np.median(ts) * 1e6), r

    def same(a, b):
        return all(np.array_equal(np.asarray(x), np.asarray(y)) for x, y in zip(a, b))

    def row(name, gpu_fn, cpu_fn, reuse_fn=None):
        g_us, g = timed(gpu_fn)
        c_us, c = timed(cpu_fn)
        assert same(g, c), name
        out[name] = {"gpu_us": round(g_us, 1), "cpu_us": round(c_us, 1), "gpu_over_cpu": round(g_us / c_us, 2), "nmatches": int(g[0])}
        if reuse_fn is not None:      # the searched frame uploaded once (vsg_frame_create) and reused, as one Track() could
            r_us, r = timed(reuse_fn)
            assert same(r, c), name
            out[name]["gpu_us_frame_reused"] = round(r_us, 1)

    f32 = lambda v: float(np.float32(v))  # noqa: E731
    _, sigma2, inv_sigma2 = sc.sigma_tables()
    # SearchByProjection(F, vpMapPoints) — a local map of 5 x the frame's features
    fd = sc.frame_data(ka, da, stereo_seed=5)
    pts, desc, occ = sc.track_points(fd, np.concatenate([kb] * 5), np.concatenate([db] * 5), (9, 5), 21, True)
    m = ORBmatcher(0.8, True, device=device)
    row("SearchByProjection(F, vpMapPoints) [%d points]" % len(pts),
        lambda: m.SearchByProjectionMap(m.frame(fd), occ, pts, desc, 3.0, False, 40.0),
        lambda: orc.search_by_projection_map(fd.view, occ, pts, desc, 3.0, False, 40.0, f32(0.8)),
        (lambda fr: lambda: m.SearchByProjectionMap(fr, occ, pts, desc, 3.0, False, 40.0))(m.frame(fd)))
    m.close()
    # SearchByProjection(Cur, Last)
    m = ORBmatcher(0.9, True, device=device)
    ppts, pdesc, pocc = sc.proj_points(fd, kb, db, (9, 5), 4)
    fr_fd = m.frame(fd)
    row("SearchByProjection(Cur, Last)", lambda: m.SearchByProjectionLast(m.frame(fd), pocc, ppts, pdesc, 15.0, 0),
        lambda: orc.search_by_projection_last(fd.view, pocc, ppts, pdesc, 15.0, 0, True),
        lambda: m.SearchByProjectionLast(fr_fd, pocc, ppts, pdesc, 15.0, 0))
    # SearchByProjection(Cur, KF, sAlreadyFound)
    spts = sc.search_points(kb, (9, 5), 3)
    socc = (rng.random(fd.n) < 0.1).astype(np.uint8)
    row("SearchByProjection(Cur, KF, sAlreadyFound)", lambda: m.SearchByProjectionReloc(m.frame(fd), socc, spts, db, 10.0, 100),
        lambda: orc.search_by_projection_reloc(fd.view, socc, spts, db, 10.0, 100, True),
        lambda: m.SearchByProjectionReloc(fr_fd, socc, spts, db, 10.0, 100))
    # SearchForInitialization (mpIniORBextractor-sized frames)
    ia, ida, ib, idb = sc.two_frames(orc, nfeat=2000)
    f1, f2 = sc.frame_data(ia, ida), sc.frame_data(ib, idb)
    prev0 = np.stack([ia["x"], ia["y"]], 1).astype(np.float32)
    row("SearchForInitialization [%d features]" % len(ia), lambda: m.SearchForInitialization(f1, m.frame(f2), prev0.copy(), 100),
        lambda: orc.search_for_initialization(f1.view, f2.view, prev0.copy(), 100, f32(0.9), True))
    m.close()
    # SearchByBoW(KF, F) / (KF, KF)
    m = ORBmatcher(0.7, True, device=device)
    kf, f = sc.frame_data(kb, db), sc.frame_data(ka, da)
    valid = (rng.random(kf.n) < 0.85).astype(np.uint8)
    valid2 = (rng.random(f.n) < 0.85).astype(np.uint8)
    kfv, ffv = sc.feature_vector(db, 24), sc.feature_vector(da, 24)
    row("SearchByBoW(KF, F)", lambda: m.SearchByBoW(kf, valid, f, kfv, ffv), lambda: orc.search_by_bow(kf.view, valid, f.view, kfv, ffv, f32(0.7), True))
    row("SearchByBoW(KF, KF)", lambda: m.SearchByBoWKF(kf, valid, f, valid2, kfv, ffv),
        lambda: orc.search_by_bow_kf(kf.view, valid, f.view, valid2, kfv, ffv, f32(0.7), True))
    m.close()
    # Sim3 projections, Fuse x 2, SearchBySim3, SearchForTriangulation
    m = ORBmatcher(0.6, True, device=device)
    fd0 = sc.frame_data(ka, da)
    matched = (rng.random(fd0.n) < 0.2).astype(np.uint8)
    spts5 = sc.search_points(kb, (9, 5), 5)
    row("SearchByProjection(KF, Scw, vpPoints)", lambda: m.SearchByProjectionSim3(m.frame(fd0), matched, spts5, db, 8, 1.0),
        lambda: orc.search_by_projection_sim3(fd0.view, matched, spts5, db, 8, f32(1.0)))
    fpts = sc.search_points(kb, (9, 5), 7, sigma=1.5)
    row("Fuse(KF, vpMapPoints) search", lambda: m.FuseSearch(m.frame(fd), fpts, db, 3.0, inv_sigma2, sim3_variant=False),
        lambda: orc.fuse_search(fd.view, fpts, db, 3.0, inv_sigma2, 0))
    row("Fuse(KF, Scw, vpPoints) search", lambda: m.FuseSearch(m.frame(fd0), fpts, db, 3.0, inv_sigma2, sim3_variant=True),
        lambda: orc.fuse_search(fd0.view, fpts, db, 3.0, inv_sigma2, 1))
    g1, g2 = sc.frame_data(ka, da), sc.frame_data(kb, db)
    p1, p2 = sc.search_points(ka, (-9, -5), 9), sc.search_points(kb, (9, 5), 10)
    row("SearchBySim3", lambda: m.SearchBySim3(m.frame(g1), m.frame(g2), p1, da, p2, db, 7.5),
        lambda: orc.search_by_sim3(g1.view, g2.view, p1, da, p2, db, 7.5))
    ta, tda, tb, tdb = sc.two_frames(orc, shift=(9, 1))
    k1, k2 = sc.frame_data(ta, tda, stereo_seed=2), sc.frame_data(tb, tdb, stereo_seed=3)
    h1, h2 = (rng.random(k1.n) < 0.3).astype(np.uint8), (rng.random(k2.n) < 0.3).astype(np.uint8)
    fv1, fv2 = sc.feature_vector(tda, 24), sc.feature_vector(tdb, 24)
    f12, ep = sc.translation_f12((9, 1)), np.array([300.0, 200.0], np.float32)
    row("SearchForTriangulation", lambda: m.SearchForTriangulation(k1, h1, k2, h2, fv1, fv2, f12, ep, sigma2, False, False),
        lambda: orc.search_for_triangulation(k1.view, h1, k2.view, h2, fv1, fv2, False, False, f12, ep, sigma2, True))
    m.close()
    return out


def sparse_frames_extras(torch, device):
    """The same pipeline on frames with a realistic corner density.  The benchmark frames (SURVEY 8d) are deliberately
    corner-rich — about 16 % of their pixels are FAST corners at threshold 20, 25 k candidates per frame — the worst case for
    the FAST kernel's strength arithmetic; indoor camera frames have a few per cent.  These frames: heavily smoothed noise
    plus 12 rectangles, ~1000 keypoints still found.  Device-resident batch of 256, CUDA events, per-stage times."""
    import numpy as np
    from visual_sgraphs_b200.extractor import ORBextractor
    rng = np.random.default_rng(99)
    try:
        from scipy.ndimage import gaussian_filter
    except Exception:  # noqa: BLE001
        return {"skipped": "scipy missing"}
    base = []
    for i in range(16):
        img = gaussian_filter(rng.random((H, W)).astype(np.float32), 6.0)
        img = (img - img.min()) / (img.max() - img.min()) * 255.0
        for _ in range(12):
            x0, y0 = int(rng.integers(0, W - 90)), int(rng.integers(0, H - 90))
            w, h = int(rng.integers(10, 90)), int(rng.integers(10, 90))
            img[y0:y0 + h, x0:x0 + w] = float(rng.integers(0, 256))
        base.append(np.clip(img + rng.normal(0, 1.0, img.shape), 0, 255).astype(np.uint8))
    B = 256
    fr = np.stack([np.roll(base[i % 16], (3 * (i // 16), 5 * (i // 16)), (0, 1)) for i in range(B)])
    d_frames = torch.from_numpy(fr).cuda()
    ex = ORBextractor(NFEAT, SCALE, NLEVELS, INI_TH, MIN_TH, device=device, max_batch=B)
    cap = ex.max_keypoints(W, H)
    kps = torch.zeros((B, cap, 28), dtype=torch.uint8, device="cuda")
    desc = torch.zeros((B, cap, 32), dtype=torch.uint8, device="cuda")
    n = torch.zeros(B, dtype=torch.int32, device="cuda")
    mono = torch.zeros(B, dtype=torch.int32, device="cuda")
    st = torch.cuda.ExternalStream(ex.stream(), device=device)
    for _ in range(3):
        ex.extract_batch_dev(d_frames, kps, desc, n, mono)
    ex.sync()
    ex.profile(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(5):
        ex.extract_batch_dev(d_frames, kps, desc, n, mono)
    e1.record(st)
    ex.sync()
    ms = e0.elapsed_time(e1) / 5
    stage_ms, runs = ex.stage_ms()
    ex.profile(False)
    cands = sum(len(ex.candidates(l, frame=0)) for l in range(NLEVELS))
    out = {"frames_per_s": B / (ms * 1e-3), "ms_per_256_frames": ms, "keypoints_per_frame": float(n.float().mean().item()),
           "fast_candidates_frame0": int(cands), "stages_ms": {k: v / max(runs, 1) for k, v in stage_ms.items()},
           "note": "the FAST kernel computes every pixel's strength regardless of content: its time is the same as on the corner-rich "
                   "benchmark frames; the oct-tree and the compaction see fewer candidates"}
    ex.close()
    return out


def main():
    reserve_stdout_for_the_json_line()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=512, help="frames per step per GPU")
    ap.add_argument("--no-extras", action="store_true", help="skip the matching and cpu-baseline extras")
    ap.add_argument("--no-stage-profile", action="store_true", help="(experiments) no per-stage events in the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of --impl ours; the reference arm only times the CPU extractor")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist

    from visual_sgraphs_b200._lib import load
    from visual_sgraphs_b200.extractor import ORBextractor

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = load()
    B, K, Wm = args.batch, args.steps, max(args.warmup, 3)

    # ---- workload: B distinct frames per rank, pinned on the host and resident in HBM ----
    host_frames = torch.from_numpy(make_frames(B, 1000 + 100000 * rank)).pin_memory()
    dev_frames = host_frames.cuda(non_blocking=False)
    ex = ORBextractor(NFEAT, SCALE, NLEVELS, INI_TH, MIN_TH, device=local_rank, max_batch=B)
    cap = ex.max_keypoints(W, H)
    kps_d = torch.zeros((B, cap, 28), dtype=torch.uint8, device="cuda")
    desc_d = torch.zeros((B, cap, 32), dtype=torch.uint8, device="cuda")
    n_d = torch.zeros(B, dtype=torch.int32, device="cuda")
    mono_d = torch.zeros(B, dtype=torch.int32, device="cuda")
    stream = torch.cuda.ExternalStream(ex.stream(), device=local_rank)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput (value) ----
    for _ in range(Wm):
        ex.extract_batch_dev(dev_frames, kps_d, desc_d, n_d, mono_d)
    ex.sync()
    sampler = ClockSampler(local_rank)
    ex.profile(not args.no_stage_profile)
    launches0 = lib.vsg_launch_count()
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(K):
        ex.extract_batch_dev(dev_frames, kps_d, desc_d, n_d, mono_d)
    e1.record(stream)
    ex.sync()
    barrier()
    clocks = sampler.result()
    launches = lib.vsg_launch_count() - launches0
    elapsed_ms = e0.elapsed_time(e1)
    stage_ms, runs = ex.stage_ms()
    ex.profile(False)
    n_kp_mean = float(n_d.float().mean().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, kps_d, desc_d, n_d, mono_d)

    # ---- end to end through the host-pointer C-ABI call (pinned frames in, pinned results out) ----
    # Two handles driven by two host threads, each taking half of the step's frames (every call is itself a chunked
    # three-stream pipeline of 128-frame chunks), so that the copies of one call overlap the kernels of the other — the
    # way a sequence driver would run it.  Measured on the B200 (chunk 128): 1 / 2 / 4 handles -> 102 / 124 / 121 k
    # frames/s; 64-frame chunks cap the rate at 117 k whatever the number of handles (small launches are less efficient).
    from visual_sgraphs_b200._lib import check, ptr
    host_np = host_frames.numpy()
    # handles (= host threads) sharing a step: three keep the copy engines and the SMs busier than two (N = 1: 144 -> 148 k,
    # N = 2: 287 -> 299 k frames/s) as long as every thread has a host core to itself
    nh_default = 3 if 3 * world <= host_threads() else 2
    nh = max(1, min(int(os.environ.get("VSG_E2E_HANDLES", str(nh_default))), B))
    alternate = os.environ.get("VSG_E2E_MODE", "split") == "alternate"      # whole steps round-robin over the handles
    cuts = [B * i // nh for i in range(nh + 1)]
    parts = [(0, B)] * nh if alternate else [(cuts[i], cuts[i + 1]) for i in range(nh)]
    handles = [ORBextractor(NFEAT, SCALE, NLEVELS, INI_TH, MIN_TH, device=local_rank, max_batch=e - b) for b, e in parts]
    outs = []
    for b, e in parts:
        kp = torch.zeros((e - b, cap, 28), dtype=torch.uint8).pin_memory()
        de = torch.zeros((e - b, cap, 32), dtype=torch.uint8).pin_memory()
        outs.append((kp, de, np.zeros(e - b, np.int32), np.zeros(e - b, np.int32)))

    def e2e_part(i):
        b, e = parts[i]
        kp, de, nn, mm = outs[i]
        check(lib.vsg_extract_batch(handles[i]._h, ptr(host_np[b:e]), e - b, W, H, W, W * H, 0, 0, ptr(kp), ptr(de), cap,
                                    ptr(nn), ptr(mm)))

    def e2e_worker(i, steps):
        for k in range(steps):
            if not alternate or k % nh == i:
                e2e_part(i)

    def e2e_run(steps):
        # each handle streams its half of every step back to back; the halves are not re-synchronised between steps
        ths = [threading.Thread(target=e2e_worker, args=(i, steps)) for i in range(len(parts))]
        for t in ths:
            t.start()
        for t in ths:
            t.join()

    e2e_run(2)
    barrier()
    launches_e2e0 = lib.vsg_launch_count()
    # K steps, three times over; the median run is reported (host threads and the PCIe link make single runs of a few
    # tens of milliseconds noisy), all three are listed in e2e.runs_ms_per_step
    e2e_runs = []
    for _ in range(3):
        t0 = time.perf_counter()
        e2e_run(K)
        torch.cuda.synchronize()
        e2e_runs.append(time.perf_counter() - t0)
        barrier()
    e2e_s = sorted(e2e_runs)[1]
    # the e2e results must be the same keypoints the device-resident path produced
    n_first = int(n_d[0].item())
    assert outs[0][2][0] == n_first, (outs[0][2][0], n_first)
    assert bytes(outs[0][0][0, :n_first].numpy().tobytes()) == bytes(kps_d[0, :n_first].cpu().numpy().tobytes())

    # the copy ceiling of this box at this N, measured now: every rank moves one step's input (pinned -> device) and one step's
    # results (device -> pinned) with plain cudaMemcpyAsync on two streams, all ranks at once, no kernels (tools/micro/h2d_all.py
    # is the stand-alone form).  e2e cannot exceed it; profiles/r02_h2d_ceiling.md has the N = 1..8 table.
    res_bytes = B * cap * 60 + 8 * B
    res_d = torch.empty(res_bytes, dtype=torch.uint8, device="cuda")
    res_h = torch.empty(res_bytes, dtype=torch.uint8).pin_memory()
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()

    def copy_step():
        with torch.cuda.stream(s_in):
            dev_frames.copy_(host_frames, non_blocking=True)
        with torch.cuda.stream(s_out):
            res_h.copy_(res_d, non_blocking=True)

    for _ in range(3):
        copy_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(10):
        copy_step()
    torch.cuda.synchronize()
    copy_s = (time.perf_counter() - t0) / 10
    barrier()
    del res_d, res_h

    times = torch.tensor([elapsed_ms, e2e_s * 1e3, copy_s * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    elapsed_ms, e2e_ms, copy_ms = float(times[0]), float(times[1]), float(times[2])
    # the sharded matcher paths (C5 train-sharded kNN-2, C3 map-sharded SearchByProjection) at this N, every rank taking part
    sharded_block = None
    if not args.no_extras:
        for hnd in handles:
            hnd.close()
        del kps_d, desc_d
        sharded_block = sharded_matching_extras(torch, dist, local_rank, rank, world)

    if rank == 0:
        frames_total = world * B * K
        value = frames_total / (elapsed_ms * 1e-3)
        tc_min = int(os.environ.get("VSG_BLUR_TC", "16") or 0)
        tc_blur = 0 < tc_min <= B                    # batches this large blur on the tensor cores (csrc/blur_tc.cu), a stage of its own
        fused = os.environ.get("VSG_FUSE_FAST_BLUR", "1") != "0" and not tc_blur
        stages_bytes, b_frame = algorithmic_bytes(W, H, n_kp_mean, fused)
        kernel_of = {"fast": "fast_blur_kernel" if fused else "fast_kernel", "blur": "blur_tc_kernel" if tc_blur else "blur_kernel",
                     "pyramid": "resize_kernel", "describe": "describe_kernel", "octree": "octree_kernel"}
        what_of = {"fast_blur_kernel": "FAST cells + Gaussian blur in one grid", "fast_kernel": "FAST-9/16 cells, threshold retry, 3x3 NMS",
                   "blur_tc_kernel": "7x7 Gaussian blur as banded u8 GEMMs on tcgen05", "blur_kernel": "7x7 Gaussian blur",
                   "resize_kernel": "pyramid levels, one launch each", "describe_kernel": "IC_Angle + rBRIEF", "octree_kernel": "DistributeOctTree"}
        peak, peak_src = measured_peaks()
        dominant = max(stage_ms, key=lambda k: stage_ms[k])
        roof_stage = dominant if stages_bytes[dominant] > 0 else "fast"
        dur_ms = stage_ms[roof_stage] / max(runs, 1) if runs else elapsed_ms / K
        achieved = stages_bytes[roof_stage] * B / (dur_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": elapsed_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": workload_config(B), "keypoints_per_frame": n_kp_mean,
            "timed_region_s": elapsed_ms * 1e-3,
            "clocks": clocks,
            "e2e": {"value": frames_total / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": B * W * H,
                    "d2h_bytes_per_step": B * cap * 60 + 8 * B, "ms_per_step": e2e_ms / K,
                    "runs_ms_per_step": [round(1e3 * t / K, 4) for t in e2e_runs], "reported": "median of 3 runs of K steps",
                    "copy_ceiling": {"value": world * B / (copy_ms * 1e-3), "unit": UNIT, "h2d_GBs_aggregate": world * B * W * H / (copy_ms * 1e-3) / 1e9,
                                     "what": "the same bytes per step with plain cudaMemcpyAsync (H2D + D2H concurrently) on all ranks at once, no kernels",
                                     "e2e_frac": (frames_total / (e2e_ms * 1e-3)) / (world * B / (copy_ms * 1e-3))}},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "%s (%s)" % (kernel_of[roof_stage], what_of[kernel_of[roof_stage]]),
                         "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak,
                         "traffic": ncu_traffic(kernel_of[roof_stage], B),
                         "pipes": ncu_pipes(kernel_of[roof_stage]),
                         "traffic_note": "bytes per launch, from the committed ncu --set full capture (profiles/ncu_traffic.json), scaled to this batch if the capture used another",
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_frame": stages_bytes[roof_stage], "launch_ms": dur_ms,
                         "dominant_stage_by_time": dominant,
                         "note": "FAST is HBM-bound by bytes but ALU-pipe bound in practice: its packed min/max alone need 1.13 ms per 512 frames "
                                 "at 100 % of the pipe (`pipes` = the committed ncu capture; DESIGN.md section 4)"},
            "stages_ms_per_step": {k: v / max(runs, 1) for k, v in stage_ms.items()},
            # every stage against the same byte roofline (SURVEY 8(d) bytes x frames / its CUDA-event time)
            "stages_hbm": {k: {"kernel": kernel_of[k], "algorithmic_bytes_per_frame": stages_bytes[k],
                               "achieved_gbs": stages_bytes[k] * B / (stage_ms[k] / max(runs, 1) * 1e-3) / 1e9,
                               "frac": stages_bytes[k] * B / (stage_ms[k] / max(runs, 1) * 1e-3) / 1e9 / peak}
                           for k in stage_ms if stages_bytes.get(k, 0) > 0 and stage_ms[k] > 0 and runs},
            "pipeline_hbm": {"algorithmic_bytes_per_frame": b_frame,
                             "achieved_gbs": b_frame * B * K / (elapsed_ms * 1e-3) / 1e9,
                             "frac": b_frame * B * K / (elapsed_ms * 1e-3) / 1e9 / peak},
        }
        if sharded_block is not None:
            line["matching_sharded"] = sharded_block
        if world == 1 and not args.no_extras:
            cores = host_threads()
            nfr = 256 * cores                       # ~10 s of CPU work on all host threads
            kind, v_all, secs_all, _ = cpu_throughput(nfr, cores)
            _, v_one, _, _ = cpu_throughput(96, 1)
            line["cpu_baseline"] = {"value": v_all, "unit": UNIT, "cores": cores, "kind": kind,
                                    "sample": "%d frames of the same workload, %d threads (one extractor per thread), %.1f s" %
                                              (nfr, cores, secs_all),
                                    "single_thread_value": v_one}
            line["single_frame_latency"] = latency_extras(torch, lib, local_rank)
            line["matching"] = matching_extras(torch, local_rank)
            line["matching_methods"] = matching_methods_extras(local_rank)
            line["realistic_corner_density"] = sparse_frames_extras(torch, local_rank)
            line["other_configs"] = other_config_extras(torch, lib, local_rank)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
