"""LocalMapping::CreateNewMapPoints' loop of SearchForTriangulation calls over a keyframe's neighbours, on the
matching_methods scenario of bench.py: two related 640x480 frames with ~1000 features, feature vectors
sc.feature_vector(desc, 24).  KF1 is frame A with about half of its features holding a map point; each neighbour is frame B
with 2% of its descriptor bits flipped (feature vector rebuilt from the flipped descriptors).

1. Through the C ABI, at 1, 10 and 30 neighbours, two forms of a stand-in loop in which every matched KF1 feature gets a
   map point after its neighbour's search: the loop of vsg_search_for_triangulation calls, and one
   vsg_triangulation_candidates_multi call plus a vsg_triangulation_resolve per neighbour.  The two forms must give the
   same pair lists.  Median and p10 / p90 of --reps runs of host wall time, the forms alternating.
2. With --parent-lib, the single-target calls of bench.py's matching_methods with this build's library and the given one
   (tools/micro/bow_candidates.py's comparison, SearchForTriangulation among them).
3. The card's name, power limit and SM clock, read before and after.

  python tools/micro/triangulation_neighbours.py [--reps 60] [--parent-lib PATH] [--rounds 8] [--out results.json]
"""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np  # noqa: E402

from bow_candidates import compare_singles, featvec_args, gpu_info, timed_pair  # noqa: E402
from oracle import oracle as orc  # noqa: E402
from tests import match_scenarios as sc  # noqa: E402
from visual_sgraphs_b200 import _lib  # noqa: E402
from visual_sgraphs_b200._lib import TriangulationTarget, check, ptr  # noqa: E402


def neighbours(keys, desc, n, seed):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        flips = (rng.random(desc.shape) < 0.02) * rng.integers(1, 256, desc.shape)
        d = (desc ^ flips).astype(np.uint8)
        out.append((sc.frame_data(keys, d, stereo_seed=3), (rng.random(len(keys)) < 0.3).astype(np.uint8), sc.feature_vector(d, 24)))
    return out


def loop_against_batch(reps):
    from visual_sgraphs_b200.matcher import ORBmatcher, _bow_side
    L = _lib.load()
    m = ORBmatcher(0.6, True)
    ka, da, kb, db = sc.two_frames(orc, shift=(9, 1))
    k1 = sc.frame_data(ka, da, stereo_seed=2)
    h1_start = (np.random.default_rng(5).random(k1.n) < 0.5).astype(np.uint8)
    fv1 = sc.feature_vector(da, 24)
    f12, ep = sc.translation_f12((9, 1)).astype(np.float32), np.array([300.0, 200.0], np.float32)
    _, sigma2, _ = sc.sigma_tables()
    sigma2 = np.ascontiguousarray(sigma2, np.float32)
    rows = []
    for T in (1, 10, 30):
        targets = neighbours(kb, db, T, 400 + T)
        keep = []
        h1 = h1_start.copy()
        K1 = _bow_side(k1, h1, fv1, keep)               # reads h1 as it is at the call
        tgs = [TriangulationTarget(_bow_side(d, v, fv, keep), (C.c_float * 9)(*f12), (C.c_float * 2)(*ep), ptr(sigma2))
               for d, v, fv in targets]
        table = (C.c_void_p * T)(*[C.addressof(t) for t in tgs])
        best = np.zeros((T, k1.n), np.int32)
        m12 = np.zeros(k1.n, np.int32)
        nm = C.c_int(0)
        pairs = {"loop": [], "batch": []}

        def loop():
            h1[:] = h1_start
            pairs["loop"] = []
            for d, v, fv in targets:
                check(L.vsg_search_for_triangulation(m._h, C.byref(k1.view), ptr(h1), C.byref(d.view), ptr(v), *featvec_args(fv1),
                                                     *featvec_args(fv), 0, 0, ptr(f12), ptr(ep), ptr(sigma2), 1, ptr(m12), C.byref(nm)))
                pairs["loop"].append(m12.copy())
                h1[m12 >= 0] = 1                        # the stand-in triangulation
        def batch():
            h1[:] = h1_start
            pairs["batch"] = []
            check(L.vsg_triangulation_candidates_multi(m._h, C.byref(K1), T, table, 0, 0, ptr(best)))
            for t, (d, _, _) in enumerate(targets):
                check(L.vsg_triangulation_resolve(C.byref(k1.view), C.byref(d.view), ptr(h1), ptr(best[t]), 1, ptr(m12), C.byref(nm)))
                pairs["batch"].append(m12.copy())
                h1[m12 >= 0] = 1

        (lu, lp), (bu, bp) = timed_pair(loop, batch, reps)
        assert all(np.array_equal(a, b) for a, b in zip(pairs["loop"], pairs["batch"])), "%d neighbours: results differ" % T
        npairs = sum(int((p >= 0).sum()) for p in pairs["batch"])
        row = dict(neighbours=T, loop_us=lu, loop_p10_p90=lp, batch_us=bu, batch_p10_p90=bp, speedup=lu / bu, pairs=npairs)
        rows.append(row)
        print("%2d neighbours: loop %8.1f us (p10-p90 %.1f-%.1f)   batch %8.1f us (p10-p90 %.1f-%.1f)   x%.2f   %d pairs" % (
            T, lu, *lp, bu, *bp, row["speedup"], npairs), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=60)
    ap.add_argument("--parent-lib", help="libvsg_cuda.so of the parent commit, for the single-call comparison")
    ap.add_argument("--rounds", type=int, default=8)
    ap.add_argument("--out", help="also write the results as JSON to this file")
    args = ap.parse_args()
    if _lib.load().vsg_device_count() < 1:
        sys.exit("triangulation_neighbours: no CUDA device")
    res = dict(gpu=gpu_info(), reps=args.reps)
    res["rows"] = loop_against_batch(args.reps)
    if args.parent_lib:
        res["singles"] = compare_singles(args.parent_lib, args.rounds, max(args.reps, 100))
    res["gpu_after"] = gpu_info()
    print(res["gpu"], "|", res["gpu_after"])
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
