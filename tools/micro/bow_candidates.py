"""The BoW candidate loops of relocalisation (Tracking::Relocalization, one frame against many keyframes) and loop detection
(LoopClosing::DetectCommonRegionsFromBoW, one keyframe against many) on the matching_methods scenario of bench.py: two
related 640x480 frames with ~1000 features, feature vectors sc.feature_vector(desc, 24).  The targets are copies of the
other frame with 2% of the descriptor bits flipped (feature vectors rebuilt from the flipped descriptors).

1. Through the C ABI, the loop of single-target calls (vsg_search_by_bow_2cam / vsg_search_by_bow_kf) against one
   vsg_search_by_bow_multi / vsg_search_by_bow_kf_multi call at 1, 10 and 33 targets, alternating the two; the results must
   be equal.  Median and p10 / p90 of --reps calls of host wall time (each call ends with a stream synchronise).
2. With --parent-lib, the single-target calls bench.py times (SearchByBoW(KF, F), SearchByBoW(KF, KF),
   SearchForTriangulation) with this build's library and with the given one, in --rounds alternating child processes
   (VSG_LIB_PATH selects the library); each number is the median over the rounds of the per-round medians.
3. The card's name, power limit and SM clock, read before and after.

  python tools/micro/bow_candidates.py [--reps 60] [--parent-lib PATH] [--rounds 8] [--out results.json]
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
from tests import match_scenarios as sc  # noqa: E402
from visual_sgraphs_b200 import _lib  # noqa: E402
from visual_sgraphs_b200._lib import check, ptr  # noqa: E402

NNRATIO = 0.7   # bench.py's matching_methods matcher for the BoW rows


def gpu_info():
    try:
        q = "name,power.limit,clocks.sm,clocks.max.sm"
        return subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return "nvidia-smi unavailable: %s" % e


def scenario():
    """bench.py matching_methods_extras: the BoW rows' frames, flags and feature vectors, and the triangulation pair."""
    ka, da, kb, db = sc.two_frames(orc)
    rng = np.random.default_rng(5)
    rng.random(len(ka))                         # the draw bench.py makes before its BoW rows
    kf, f = sc.frame_data(kb, db), sc.frame_data(ka, da)
    valid = (rng.random(kf.n) < 0.85).astype(np.uint8)
    valid2 = (rng.random(f.n) < 0.85).astype(np.uint8)
    return ka, da, kb, db, kf, f, valid, valid2, rng


def perturbed(keys, desc, ntargets, seed):
    """ntargets keyframes: desc with 2% of the bits flipped, flags for 85% of the features, feature vectors rebuilt."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(ntargets):
        flips = (rng.random(desc.shape) < 0.02) * rng.integers(1, 256, desc.shape)
        d = (desc ^ flips).astype(np.uint8)
        out.append((sc.frame_data(keys, d), (rng.random(len(keys)) < 0.85).astype(np.uint8), sc.feature_vector(d, 24)))
    return out


def featvec_args(fv):
    n, p, i = fv
    return [len(n), ptr(n), ptr(p), ptr(i)]


def timed_pair(fa, fb, reps):
    for _ in range(10):                         # warm-up: buffers grown, modules loaded
        fa(), fb()
    sa, sb = [], []
    for _ in range(reps):                       # alternate the two forms
        t0 = time.perf_counter(); fa(); sa.append(time.perf_counter() - t0)
        t0 = time.perf_counter(); fb(); sb.append(time.perf_counter() - t0)
    stats = lambda s: (float(np.median(s) * 1e6), [float(np.percentile(s, q) * 1e6) for q in (10, 90)])  # noqa: E731
    return stats(sa), stats(sb)


def loops_against_multi(reps):
    from visual_sgraphs_b200.matcher import ORBmatcher, _bow_side, _side_table
    L = _lib.load()
    ka, da, kb, db, kf, f, valid, valid2, _ = scenario()
    m = ORBmatcher(NNRATIO, True)
    ffv, kfv = sc.feature_vector(da, 24), sc.feature_vector(db, 24)
    rows = []
    for T in (1, 10, 33):
        for form in ("KF-F", "KF-KF"):
            # KF-F: keyframes from frame B against frame A; KF-KF: frame B's keyframe against keyframes from frame A
            targets = perturbed(kb, db, T, 100 + T) if form == "KF-F" else perturbed(ka, da, T, 200 + T)
            keep = []
            sides = [_bow_side(d, v, fv, keep) for d, v, fv in targets]
            tab = _side_table(sides)
            n_out = f.n if form == "KF-F" else kf.n
            out_loop, out_multi = np.zeros((T, n_out), np.int32), np.zeros((T, n_out), np.int32)
            nm_loop, nm_multi = np.zeros(T, np.int32), np.zeros(T, np.int32)
            nm1 = C.c_int(0)
            if form == "KF-F":
                F = _bow_side(f, None, ffv, keep)
                args = [(C.byref(d.view), ptr(v), C.byref(f.view), -1, *featvec_args(fv), *featvec_args(ffv), C.c_float(NNRATIO), 1,
                         ptr(out_loop[t]), C.byref(nm1)) for t, (d, v, fv) in enumerate(targets)]
                single, multi_args = L.vsg_search_by_bow_2cam, (m._h, T, tab, C.byref(F), -1, C.c_float(NNRATIO), 1,
                                                               ptr(out_multi), ptr(nm_multi))
                multi_fn = L.vsg_search_by_bow_multi
            else:
                K1 = _bow_side(kf, valid, kfv, keep)
                args = [(C.byref(kf.view), ptr(valid), C.byref(d.view), ptr(v), *featvec_args(kfv), *featvec_args(fv),
                         C.c_float(NNRATIO), 1, ptr(out_loop[t]), C.byref(nm1)) for t, (d, v, fv) in enumerate(targets)]
                single, multi_args = L.vsg_search_by_bow_kf, (m._h, C.byref(K1), T, tab, C.c_float(NNRATIO), 1, ptr(out_multi),
                                                             ptr(nm_multi))
                multi_fn = L.vsg_search_by_bow_kf_multi

            def loop():
                for t, a in enumerate(args):
                    check(single(m._h, *a))
                    nm_loop[t] = nm1.value

            (lu, lp), (mu, mp) = timed_pair(loop, lambda: check(multi_fn(*multi_args)), reps)
            assert np.array_equal(out_loop, out_multi) and np.array_equal(nm_loop, nm_multi), "%s, %d targets: results differ" % (
                form, T)
            row = dict(form=form, targets=T, loop_us=lu, loop_p10_p90=lp, multi_us=mu, multi_p10_p90=mp, speedup=lu / mu,
                       matches_per_target=float(nm_multi.mean()))
            rows.append(row)
            print("%-5s %2d targets: loop %8.1f us (p10-p90 %.1f-%.1f)   multi %8.1f us (p10-p90 %.1f-%.1f)   x%.2f   %.0f matches "
                  "per target" % (form, T, lu, *lp, mu, *mp, row["speedup"], row["matches_per_target"]), flush=True)
    return rows


def singles(reps):
    """Child process: the single-target BoW calls of bench.py's matching_methods through the library VSG_LIB_PATH names
    (only the symbols the parent commit already has are bound).  Prints one JSON line of median microseconds."""
    L = C.CDLL(_lib.LIB_PATH)
    for name in ("vsg_matcher_create", "vsg_matcher_destroy", "vsg_search_by_bow_2cam", "vsg_search_by_bow_kf",
                 "vsg_search_for_triangulation"):
        res, argt = _lib._SIGNATURES[name]
        getattr(L, name).restype, getattr(L, name).argtypes = res, argt
    ka, da, kb, db, kf, f, valid, valid2, rng = scenario()
    kfv, ffv = sc.feature_vector(db, 24), sc.feature_vector(da, 24)
    h = C.c_void_p()
    assert L.vsg_matcher_create(0, C.byref(h)) == 0
    nm = C.c_int(0)
    out_f, out_k = np.zeros(f.n, np.int32), np.zeros(kf.n, np.int32)
    # SearchForTriangulation as bench.py sets it up
    rng.random(len(ka))
    ta, tda, tb, tdb = sc.two_frames(orc, shift=(9, 1))
    k1, k2 = sc.frame_data(ta, tda, stereo_seed=2), sc.frame_data(tb, tdb, stereo_seed=3)
    h1, h2 = (rng.random(k1.n) < 0.3).astype(np.uint8), (rng.random(k2.n) < 0.3).astype(np.uint8)
    fv1, fv2 = sc.feature_vector(tda, 24), sc.feature_vector(tdb, 24)
    f12, ep = sc.translation_f12((9, 1)).astype(np.float32).reshape(9), np.array([300.0, 200.0], np.float32)
    _, sigma2, _ = sc.sigma_tables()
    sigma2 = np.ascontiguousarray(sigma2, np.float32)
    out_t = np.zeros(k1.n, np.int32)
    calls = {
        "SearchByBoW(KF, F)": lambda: L.vsg_search_by_bow_2cam(h, C.byref(kf.view), ptr(valid), C.byref(f.view), -1, *featvec_args(kfv),
                                                               *featvec_args(ffv), C.c_float(NNRATIO), 1, ptr(out_f), C.byref(nm)),
        "SearchByBoW(KF, KF)": lambda: L.vsg_search_by_bow_kf(h, C.byref(kf.view), ptr(valid), C.byref(f.view), ptr(valid2),
                                                              *featvec_args(kfv), *featvec_args(ffv), C.c_float(NNRATIO), 1,
                                                              ptr(out_k), C.byref(nm)),
        "SearchForTriangulation": lambda: L.vsg_search_for_triangulation(h, C.byref(k1.view), ptr(h1), C.byref(k2.view), ptr(h2),
                                                                         *featvec_args(fv1), *featvec_args(fv2), 0, 0, ptr(f12),
                                                                         ptr(ep), ptr(sigma2), 1, ptr(out_t), C.byref(nm)),
    }
    res = {}
    for name, fn in calls.items():
        for _ in range(10):
            assert fn() == 0
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        res[name] = (float(np.median(ts) * 1e6), int(nm.value))
    L.vsg_matcher_destroy(h)
    print("SINGLES " + json.dumps(res), flush=True)


def compare_singles(parent_lib, rounds, reps):
    libs = {"this build": _lib.LIB_PATH, "parent": os.path.abspath(parent_lib)}
    samples = {k: [] for k in libs}
    for _ in range(rounds):                     # alternate the two libraries, one child process each
        for k, path in libs.items():
            env = dict(os.environ, VSG_LIB_PATH=path)
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--singles", "--reps", str(reps)], env=env,
                                 capture_output=True, text=True, check=True).stdout
            samples[k].append(json.loads(out.split("SINGLES ", 1)[1]))
    res = {}
    for name in samples["this build"][0]:
        row = {}
        for k in libs:
            row[k + "_us"] = float(np.median([s[name][0] for s in samples[k]]))
            row[k + "_nmatches"] = samples[k][0][name][1]
        assert row["this build_nmatches"] == row["parent_nmatches"], name
        row["ratio"] = row["this build_us"] / row["parent_us"]
        res[name] = row
        print("%-24s this build %7.1f us   parent %7.1f us   ratio %.3f   (%d matches)" % (
            name, row["this build_us"], row["parent_us"], row["ratio"], row["this build_nmatches"]), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=60)
    ap.add_argument("--parent-lib", help="libvsg_cuda.so of the parent commit, for the single-call comparison")
    ap.add_argument("--rounds", type=int, default=8)
    ap.add_argument("--singles", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--out", help="also write the results as JSON to this file")
    args = ap.parse_args()
    if args.singles:
        return singles(args.reps)
    if _lib.load().vsg_device_count() < 1:
        sys.exit("bow_candidates: no CUDA device")
    res = dict(gpu=gpu_info(), reps=args.reps)
    res["rows"] = loops_against_multi(args.reps)
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
