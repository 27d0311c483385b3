"""LocalMapping::SearchInNeighbors-shaped Fuse workload (LocalMapping.cc:764-802) at 640x480 with 1000 features: the
current keyframe's ~1000 map points are fused into 10, 20 and 30 target keyframes of ~1000 keypoints each (half of them
stereo).  Times, through the C ABI with every frame already created, the loop of single-target vsg_fuse_search calls
against one vsg_fuse_search_multi call over all targets, alternating the two, and checks that they return the same
indices.  Also times a 1-target multi call against one vsg_fuse_search.  Each number is the median of --reps calls of
host wall time around the call (each call ends with a stream synchronise).

  python tools/micro/fuse_neighbours.py [--reps 60] [--out results.json]
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


def build_targets(ka, da, kb, db, ntargets, seed):
    """Target t: frame A's keypoints moved by a per-target offset (plus 0.3 px noise, 2% descriptor bits flipped), and the
    current keyframe's map points (frame B's keypoints) projected into it."""
    rng = np.random.default_rng(seed)
    frames, pts = [], []
    for t in range(ntargets):
        off = rng.uniform(-20, 20, 2).astype(np.float32)
        keys = ka.copy()
        keys["x"] = np.clip(keys["x"] + off[0] + rng.normal(0, 0.3, len(keys)), 0, 639.9).astype(np.float32)
        keys["y"] = np.clip(keys["y"] + off[1] + rng.normal(0, 0.3, len(keys)), 0, 479.9).astype(np.float32)
        flips = (rng.random(da.shape) < 0.02) * rng.integers(1, 256, da.shape)
        frames.append(sc.frame_data(keys, (da ^ flips).astype(np.uint8), stereo_seed=seed + t if t % 2 == 0 else None))
        p = sc.search_points(kb, (9 - off[0], 5 - off[1]), seed + 100 + t, sigma=1.0)
        p["ur"] = p["u"] - 12.0
        pts.append(p)
    return frames, np.ascontiguousarray(np.stack(pts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=60)
    ap.add_argument("--out", help="also write the results as JSON to this file")
    args = ap.parse_args()
    L = _lib.load()
    if L.vsg_device_count() < 1:
        sys.exit("fuse_neighbours: no CUDA device")
    ka, da, kb, db = sc.two_frames(orc)
    _, _, inv_sigma2 = sc.sigma_tables()
    desc = np.ascontiguousarray(db)
    n = len(desc)
    m = ORBmatcher()
    res = dict(gpu=gpu_info(), points=n, reps=args.reps, rows=[])

    for T in (1, 10, 20, 30):
        fds, pts = build_targets(ka, da, kb, db, T, 1000 + T)
        frames = [m.frame(fd) for fd in fds]
        fh = (C.c_void_p * T)(*[f._h.value for f in frames])
        sig = (C.c_void_p * T)(*([inv_sigma2.ctypes.data] * T))
        out_multi = np.zeros((T, n), np.int32)
        out_loop = np.zeros((T, n), np.int32)
        nf = C.c_int(0)
        pts_t = [pts[t] for t in range(T)]
        dptr, sptr, th = ptr(desc), ptr(inv_sigma2), C.c_float(3.0)
        loop_args = [(frames[t]._h, n, ptr(pts_t[t]), dptr, th, sptr, 0, ptr(out_loop[t]), C.byref(nf)) for t in range(T)]
        multi_args = (m._h, T, fh, sig, n, ptr(pts), dptr, th, ptr(out_multi))

        def loop():
            t0 = time.perf_counter()
            for a in loop_args:
                check(L.vsg_fuse_search(m._h, *a))
            return time.perf_counter() - t0

        def multi():
            t0 = time.perf_counter()
            check(L.vsg_fuse_search_multi(*multi_args))
            return time.perf_counter() - t0

        for _ in range(10):                        # warm-up: buffers grown, modules loaded
            loop(), multi()
        samples_l, samples_m = [], []
        for _ in range(args.reps):                 # alternate the two forms
            samples_l.append(loop())
            samples_m.append(multi())
        assert np.array_equal(out_loop, out_multi), "multi-target and loop results differ at %d targets" % T
        row = dict(targets=T, loop_us=float(np.median(samples_l) * 1e6), multi_us=float(np.median(samples_m) * 1e6),
                   loop_p10_p90=[float(np.percentile(samples_l, q) * 1e6) for q in (10, 90)],
                   multi_p10_p90=[float(np.percentile(samples_m, q) * 1e6) for q in (10, 90)],
                   fused_per_target=float((out_multi >= 0).sum() / T))
        row["speedup"] = row["loop_us"] / row["multi_us"]
        res["rows"].append(row)
        print("%2d targets: loop of vsg_fuse_search %8.1f us  (p10-p90 %.1f-%.1f)   vsg_fuse_search_multi %8.1f us  "
              "(p10-p90 %.1f-%.1f)   x%.2f   %.0f fused per target" %
              (T, row["loop_us"], *row["loop_p10_p90"], row["multi_us"], *row["multi_p10_p90"], row["speedup"],
               row["fused_per_target"]), flush=True)
        for f in frames:
            f.close()
    res["gpu_after"] = gpu_info()
    print(res["gpu"])
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
