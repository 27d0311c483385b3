"""MapPoint::ComputeDistinctiveDescriptors-shaped workload (MapPoint.cc:340-417) through the C ABI: one
vsg_distinctive_descriptors call over a keyframe's map points.  Inputs: 300 / 1000 / 3000 points with seeded observation
counts from 2 to 60 (LocalMapping's two loops over a keyframe's points), and 1000 points of a uniform n = 2, 10, 32 and 100.

Times this tree's library against another build of it (--parent, e.g. the parent commit's libvsg_cuda.so, the library
VSG_LIB_PATH would load), alternating the two in one run, and checks that both return the same rows.  The parent is timed
twice per round (P and P'), so the P / P' ratio of the medians measures the spread of the comparison itself.  Each number
is the median (and p10-p90) of --reps calls of host wall time around the call (each call ends with a stream synchronise).
The kernels' device time per call comes from torch.profiler, in a separate pass of 50 calls per library.
The CPU figure is the oracle's restatement of the reference's per-point method (oracle/liborb_oracle.so), called once per
point through ctypes on the same host; the ctypes cost of a call is measured separately and reported beside it.  The card's
name, power limit and clocks are read in the same run.

  python tools/micro/distinctive_points.py --parent /path/to/parent/libvsg_cuda.so [--reps 200] [--out results.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

from oracle import oracle as orc  # noqa: E402
from visual_sgraphs_b200 import _lib  # noqa: E402


def gpu_info():
    try:
        q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
        return subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return "nvidia-smi unavailable: %s" % e


def workload(counts, seed):
    """One map point per count: a base descriptor, each observation with 2-30 % of its bits flipped."""
    rng = np.random.default_rng(seed)
    ptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    base = rng.integers(0, 256, (len(counts), 32), dtype=np.uint8)
    owner = np.repeat(np.arange(len(counts)), counts)
    rate = rng.uniform(0.02, 0.3, len(owner))[:, None]
    flips = np.packbits(rng.random((len(owner), 256)) < rate, axis=1)
    return np.ascontiguousarray(base[owner] ^ flips), ptr


class Lib:
    def __init__(self, path):
        self.L = C.CDLL(path)
        self.L.vsg_matcher_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        self.L.vsg_distinctive_descriptors.argtypes = [C.c_void_p] * 3 + [C.c_int, C.c_void_p]
        self.m = C.c_void_p()
        assert self.L.vsg_matcher_create(0, C.byref(self.m)) == 0, path

    def timed(self, desc, ptr, out):
        t0 = time.perf_counter()
        st = self.L.vsg_distinctive_descriptors(self.m, desc.ctypes.data, ptr.ctypes.data, len(out), out.ctypes.data)
        t = time.perf_counter() - t0
        assert st == 0
        return t


def kernel_us(lib, desc, ptr, out, calls=50):
    """Device time of the call's kernels (every kernel whose name holds "distinctive") per call, from torch.profiler with
    CUDA activities, in a pass of its own after the timed ones."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            lib.timed(desc, ptr, out)
    total = 0.0
    for e in prof.key_averages():
        if "distinctive" in e.key:
            total += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
    return total / calls


def stats(samples):
    return dict(median_us=float(np.median(samples) * 1e6), p10_p90_us=[float(np.percentile(samples, q) * 1e6) for q in (10, 90)])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent", required=True, help="the libvsg_cuda.so to compare with")
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--out", help="also write the results as JSON to this file")
    args = ap.parse_args()
    if _lib.load().vsg_device_count() < 1:
        sys.exit("distinctive_points: no CUDA device")
    new, parent = Lib(_lib.LIB_PATH), Lib(os.path.abspath(args.parent))
    O = orc.lib()
    res = dict(gpu=gpu_info(), reps=args.reps, library=_lib.LIB_PATH, parent=os.path.abspath(args.parent), rows=[])
    print(res["gpu"], flush=True)
    cases = [("keyframe", n, np.random.default_rng(n).integers(2, 61, n)) for n in (300, 1000, 3000)]
    cases += [("uniform n=%d" % k, 1000, np.full(1000, k)) for k in (2, 10, 32, 100)]
    for name, npts, counts in cases:
        desc, ptr = workload(counts, 17 + npts + int(counts[0]))
        out_new, out_par = np.zeros(npts, np.int32), np.zeros(npts, np.int32)
        for _ in range(10):                                    # warm-up: buffers grown, modules loaded
            new.timed(desc, ptr, out_new)
            parent.timed(desc, ptr, out_par)
        assert np.array_equal(out_new, out_par), name
        sn, sp, sp2 = [], [], []
        for _ in range(args.reps):                             # alternate: this library, the parent, the parent again
            sn.append(new.timed(desc, ptr, out_new))
            sp.append(parent.timed(desc, ptr, out_par))
            sp2.append(parent.timed(desc, ptr, out_par))
        assert np.array_equal(out_new, out_par), name
        dp = desc.ctypes.data
        t0 = time.perf_counter()                               # the oracle, one ctypes call per point
        want = [O.orc_distinctive_descriptor(C.c_void_p(dp + 32 * int(ptr[p])), int(ptr[p + 1] - ptr[p])) for p in range(npts)]
        t_orc = time.perf_counter() - t0
        t0 = time.perf_counter()                               # the same calls with n = 0: the ctypes cost alone
        for p in range(npts):
            O.orc_distinctive_descriptor(C.c_void_p(dp), 0)
        t_ctypes = time.perf_counter() - t0
        assert want == out_new.tolist(), name
        row = dict(case=name, points=npts, rows=int(ptr[-1]), new=stats(sn), parent=stats(sp), parent_again=stats(sp2),
                   oracle_loop_us=t_orc * 1e6, oracle_ctypes_us=t_ctypes * 1e6)
        row["speedup_vs_parent"] = row["parent"]["median_us"] / row["new"]["median_us"]
        row["kernel_us"] = kernel_us(new, desc, ptr, out_new)
        row["parent_kernel_us"] = kernel_us(parent, desc, ptr, out_par)
        row["parent_spread"] = row["parent"]["median_us"] / row["parent_again"]["median_us"]
        res["rows"].append(row)
        print("%-13s %5d points %6d rows: this %8.1f us (p10-p90 %.1f-%.1f)  parent %8.1f us (p10-p90 %.1f-%.1f)  x%.2f  "
              "P/P' %.3f   kernels %.1f vs %.1f us   oracle loop %9.1f us (ctypes %.1f us)" %
              (name, npts, row["rows"], row["new"]["median_us"], *row["new"]["p10_p90_us"], row["parent"]["median_us"],
               *row["parent"]["p10_p90_us"], row["speedup_vs_parent"], row["parent_spread"], row["kernel_us"], row["parent_kernel_us"], row["oracle_loop_us"],
               row["oracle_ctypes_us"]), flush=True)
    res["gpu_after"] = gpu_info()
    print(res["gpu_after"])
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
