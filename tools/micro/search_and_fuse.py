"""LoopClosing::SearchAndFuse-shaped Fuse workload (LoopClosing.cc:1994-2054) at 640x480 with 1000 features: the map
points of a loop keyframe's covisibility group (1 000, 4 000 or 12 000 of them) are fused into 1, 10, 30 or 60 corrected
keyframes of ~1000 keypoints each.  Times, through the C ABI with every frame already created, the loop of single-target
vsg_fuse_search calls (variant 1, no gates) against one vsg_fuse_search_sim3_multi call over all targets, alternating the
two, and checks that they return the same indices.  Each number is the median (and p10-p90) of --reps calls of host wall
time around the call (each call ends with a stream synchronise).  The card's name, power limit and clocks are read in the
same run.

  python tools/micro/search_and_fuse.py [--reps 60] [--out results.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np  # noqa: E402

from oracle import oracle as orc  # noqa: E402
from tests import match_scenarios as sc  # noqa: E402
from visual_sgraphs_b200 import _lib  # noqa: E402
from visual_sgraphs_b200._lib import check, ptr  # noqa: E402
from visual_sgraphs_b200.matcher import ORBmatcher  # noqa: E402


def gpu_info():
    try:
        q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
        return subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return "nvidia-smi unavailable: %s" % e


def build(ka, da, kb, db, n, ntargets, seed):
    """n map points (frame B's keypoints repeated, 2% descriptor bits flipped per copy), and ntargets keyframes: frame A's
    keypoints moved by a per-target offset (plus 0.3 px noise and 2% flipped bits), with every point projected into each."""
    rng = np.random.default_rng(seed)
    reps = -(-n // len(kb))
    desc = np.concatenate([db ^ (rng.random(db.shape) < 0.02) * rng.integers(1, 256, db.shape, dtype=np.uint8)
                           for _ in range(reps)]).astype(np.uint8)[:n]
    frames, pts = [], []
    for t in range(ntargets):
        off = rng.uniform(-20, 20, 2).astype(np.float32)
        keys = ka.copy()
        keys["x"] = np.clip(keys["x"] + off[0] + rng.normal(0, 0.3, len(keys)), 0, 639.9).astype(np.float32)
        keys["y"] = np.clip(keys["y"] + off[1] + rng.normal(0, 0.3, len(keys)), 0, 479.9).astype(np.float32)
        flips = (rng.random(da.shape) < 0.02) * rng.integers(1, 256, da.shape)
        frames.append(sc.frame_data(keys, (da ^ flips).astype(np.uint8)))
        pts.append(np.concatenate([sc.search_points(kb, (9 - off[0], 5 - off[1]), seed + 100 * t + r, sigma=1.0)
                                   for r in range(reps)])[:n])
    return frames, np.ascontiguousarray(np.stack(pts)), np.ascontiguousarray(desc)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=60)
    ap.add_argument("--out", help="also write the results as JSON to this file")
    args = ap.parse_args()
    L = _lib.load()
    if L.vsg_device_count() < 1:
        sys.exit("search_and_fuse: no CUDA device")
    ka, da, kb, db = sc.two_frames(orc)
    m = ORBmatcher()
    res = dict(gpu=gpu_info(), reps=args.reps, rows=[])
    print(res["gpu"], flush=True)
    th = C.c_float(4.0)
    for n in (1000, 4000, 12000):
        for T in (1, 10, 30, 60):
            fds, pts, desc = build(ka, da, kb, db, n, T, 7000 + 100 * T + n // 1000)
            frames = [m.frame(fd) for fd in fds]
            fh = (C.c_void_p * T)(*[f._h.value for f in frames])
            out_multi = np.zeros((T, n), np.int32)
            out_loop = np.zeros((T, n), np.int32)
            nf = C.c_int(0)
            dptr = ptr(desc)
            loop_args = [(frames[t]._h, n, ptr(pts[t]), dptr, th, None, 1, ptr(out_loop[t]), C.byref(nf)) for t in range(T)]
            multi_args = (m._h, T, fh, n, ptr(pts), dptr, th, ptr(out_multi))

            def loop():
                t0 = time.perf_counter()
                for a in loop_args:
                    check(L.vsg_fuse_search(m._h, *a))
                return time.perf_counter() - t0

            def multi():
                t0 = time.perf_counter()
                check(L.vsg_fuse_search_sim3_multi(*multi_args))
                return time.perf_counter() - t0

            for _ in range(5):                         # warm-up: buffers grown, modules loaded
                loop(), multi()
            samples_l, samples_m = [], []
            for _ in range(args.reps):                 # alternate the two forms
                samples_l.append(loop())
                samples_m.append(multi())
            assert np.array_equal(out_loop, out_multi), "one call and loop results differ at n=%d, %d targets" % (n, T)
            row = dict(points=n, targets=T, loop_us=float(np.median(samples_l) * 1e6), multi_us=float(np.median(samples_m) * 1e6),
                       loop_p10_p90=[float(np.percentile(samples_l, q) * 1e6) for q in (10, 90)],
                       multi_p10_p90=[float(np.percentile(samples_m, q) * 1e6) for q in (10, 90)],
                       found_per_target=float((out_multi >= 0).sum() / T))
            row["speedup"] = row["loop_us"] / row["multi_us"]
            res["rows"].append(row)
            print("n=%5d T=%2d: loop of vsg_fuse_search %9.1f us (p10-p90 %.1f-%.1f)   vsg_fuse_search_sim3_multi %9.1f us "
                  "(p10-p90 %.1f-%.1f)   x%.2f   %.0f found per target" %
                  (n, T, row["loop_us"], *row["loop_p10_p90"], row["multi_us"], *row["multi_p10_p90"], row["speedup"],
                   row["found_per_target"]), flush=True)
            for f in frames:
                f.close()
    res["gpu_after"] = gpu_info()
    print(res["gpu_after"])
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
