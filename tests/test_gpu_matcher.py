"""GPU parity tests for the Hamming matching kernels (bit-exact integer work) against the oracle's
DescriptorDistance and numpy restatements of the candidate scans."""
import numpy as np
import pytest

from visual_sgraphs_b200.synth import synth_descriptors, synth_query_train

pytestmark = pytest.mark.gpu

POP = np.array([bin(i).count("1") for i in range(256)], np.int32)


def hamming_matrix(q, t):
    return POP[np.bitwise_xor(q[:, None, :], t[None, :, :])].sum(-1).astype(np.int32)


def knn2_ref(q, t):
    d = hamming_matrix(q, t)
    key = d.astype(np.int64) * (1 << 32) + np.arange(t.shape[0])[None, :]
    order = np.argsort(key, axis=1, kind="stable")[:, :2]
    idx = order.astype(np.int32)
    dist = np.take_along_axis(d, order, 1)
    return idx, dist


def _matcher():
    from visual_sgraphs_b200.matcher import ORBmatcher
    return ORBmatcher()


def test_descriptor_distance_matches_oracle(oracle):
    a, b = synth_descriptors(1, 3000), synth_descriptors(2, 3000)
    b[:100] = a[:100]
    a[100] = 0
    b[100] = 255
    got = _matcher().DescriptorDistance(a, b)
    want = np.array([oracle.descriptor_distance(a[i], b[i]) for i in range(len(a))], np.int32)
    assert np.array_equal(got, want)
    assert got[0] == 0 and got[100] == 256


@pytest.mark.parametrize("nq,nt", [(1, 1), (1, 2), (7, 5), (100, 1000), (1000, 4097), (1030, 20000), (3, 0)])
def test_knn2_matches_bruteforce(nq, nt):
    q, t = synth_query_train(nq * 31 + nt, nq, max(nt, 1))
    t = t[:nt]
    if nt >= 8:
        t[3] = t[1]          # exact duplicates: ties must resolve to the lower train index
        q[0] = t[1]
    idx, dist = _matcher().knn2(q, t)
    if nt == 0:
        assert (idx == -1).all() and (dist == np.iinfo(np.int32).max).all()
        return
    widx, wdist = knn2_ref(q, t)
    if nt == 1:
        assert np.array_equal(idx[:, 0], widx[:, 0]) and np.array_equal(dist[:, 0], wdist[:, 0])
        assert (idx[:, 1] == -1).all()
        return
    assert np.array_equal(dist, wdist)
    assert np.array_equal(idx, widx)


def test_knn2_index_offset_and_merge_of_shards():
    torch = pytest.importorskip("torch")
    q, t = synth_query_train(77, 500, 6000)
    m = _matcher()
    widx, wdist = knn2_ref(q, t)
    shards = np.array_split(np.arange(6000), 4)
    dq = torch.from_numpy(q).cuda()
    parts_i = torch.zeros((4, 500, 2), dtype=torch.int32, device="cuda")
    parts_d = torch.zeros((4, 500, 2), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    for s, rows in enumerate(shards):
        dt = torch.from_numpy(t[rows]).cuda()
        torch.cuda.synchronize()
        m.knn2_dev(dq, dt, parts_i[s], parts_d[s], train_index_offset=int(rows[0]))
        m.sync()
    oi = torch.zeros((500, 2), dtype=torch.int32, device="cuda")
    od = torch.zeros((500, 2), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    m.knn2_merge_dev(parts_i, parts_d, oi, od)
    m.sync()
    assert np.array_equal(oi.cpu().numpy(), widx)
    assert np.array_equal(od.cpu().numpy(), wdist)


def window_ref(q, t, cand_ptr, cand, skip, level, init):
    nq = q.shape[0]
    out = {k: np.zeros(nq, np.int32) for k in ("best_idx", "best_dist", "second_dist", "best_level", "second_level")}
    for i in range(nq):
        bd = bd2 = init
        bi = bl = bl2 = -1
        for c in range(cand_ptr[i], cand_ptr[i + 1]):
            j = cand[c]
            if skip is not None and skip[j]:
                continue
            d = int(POP[np.bitwise_xor(q[i], t[j])].sum())
            lv = int(level[j]) if level is not None else -1
            if d < bd:
                bd2, bd, bl2, bl, bi = bd, d, bl, lv, j
            elif d < bd2:
                bl2, bd2 = lv, d
        out["best_idx"][i], out["best_dist"][i], out["second_dist"][i] = bi, bd, bd2
        out["best_level"][i], out["second_level"][i] = bl, bl2
    return out


@pytest.mark.parametrize("init", [256, np.iinfo(np.int32).max])
def test_match_window_matches_sequential_scan(init):
    rng = np.random.default_rng(5)
    q, t = synth_query_train(9, 800, 1000, related_frac=0.5)
    counts = rng.integers(0, 25, 800)
    cand_ptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    cand = rng.integers(0, 1000, cand_ptr[-1]).astype(np.int32)
    skip = (rng.random(1000) < 0.2).astype(np.uint8)
    level = rng.integers(0, 8, 1000).astype(np.int32)
    got = _matcher().match_window(q, t, cand_ptr, cand, skip, level, init)
    want = window_ref(q, t, cand_ptr, cand, skip, level, init)
    for k in want:
        assert np.array_equal(got[k], want[k]), k
    got2 = _matcher().match_window(q, t, cand_ptr, cand, None, None, init)
    want2 = window_ref(q, t, cand_ptr, cand, None, None, init)
    for k in want2:
        assert np.array_equal(got2[k], want2[k]), k


def test_distinctive_descriptors_batch(oracle):
    """vsg_distinctive_descriptors against the oracle's MapPoint::ComputeDistinctiveDescriptors restatement, for a batch
    of map points with 0 .. 1500 observations (1500 > the shared-memory staging limit)."""
    from visual_sgraphs_b200.matcher import ORBmatcher
    rng = np.random.default_rng(5)
    sizes = [0, 1, 2, 3, 5, 8, 13, 31, 32, 33, 64, 100, 257, 1500] + rng.integers(1, 40, 300).tolist()
    descs, ptr = [], [0]
    for n in sizes:
        base = rng.integers(0, 256, 32, dtype=np.uint8)
        d = np.stack([base ^ np.packbits(rng.random(256) < rng.uniform(0.02, 0.3)) for _ in range(n)]) if n else \
            np.zeros((0, 32), np.uint8)
        if n > 3:
            d[3] = d[1]
        descs.append(d)
        ptr.append(ptr[-1] + n)
    got = ORBmatcher().ComputeDistinctiveDescriptors(np.concatenate(descs), ptr)
    want = [oracle.distinctive_descriptor(d) for d in descs]
    assert got.tolist() == want


def test_knn2_ratio_filter(oracle):
    from visual_sgraphs_b200.matcher import ORBmatcher
    from visual_sgraphs_b200.synth import synth_query_train
    q, t = synth_query_train(9, 300, 2000)
    m = ORBmatcher()
    match, dist = m.knn2_ratio(q, t, 0.7)
    idx, d = m.knn2(q, t)
    want = np.where(d[:, 0].astype(np.float32) < d[:, 1].astype(np.float32).astype(np.float64) * np.float64(np.float32(0.7)), idx[:, 0], -1)
    assert np.array_equal(match, want) and np.array_equal(dist, d[:, 0])
    assert (match >= 0).sum() > 10
    one, _ = m.knn2_ratio(q[:5], t[:1], 0.7)          # fewer than two neighbours: (*it).size() >= 2 fails
    assert (one == -1).all()


def test_bow_transform(oracle):
    """vsg_bow_transform (GPU tree walk) against the oracle's restatement of DBoW2's transform, and the BowVector /
    FeatureVector bookkeeping of Vocabulary.transform against a direct restatement of TemplatedVocabulary.h:1139-1205."""
    from tests import match_scenarios as sc
    from visual_sgraphs_b200.matcher import ORBmatcher
    from visual_sgraphs_b200.vocabulary import Vocabulary
    voc = sc.synthetic_vocabulary(4, k=10, levels=4)
    m = ORBmatcher()
    V = Vocabulary(m, voc["child_ptr"], voc["child_idx"], voc["node_desc"], voc["word_id"], voc["weight"], voc["levels"])
    rng = np.random.default_rng(2)
    nd = voc["node_desc"]
    feats = np.stack([nd[rng.integers(1, len(nd))] ^ np.packbits(rng.random(256) < 0.08) for _ in range(2000)])
    feats[0] = nd[voc["child_idx"][voc["child_ptr"][1]]]
    for levelsup in (4, 2, 1, 0, 6):
        leaf, nid = V.walk(feats, levelsup)
        wleaf, wnid = oracle.bow_transform(voc["child_ptr"], voc["child_idx"], nd, voc["levels"], feats, levelsup)
        assert np.array_equal(leaf, wleaf) and np.array_equal(nid, wnid), levelsup
    bow, (nodes, ptr_, idx) = V.transform(feats, 2)
    wleaf, wnid = oracle.bow_transform(voc["child_ptr"], voc["child_idx"], nd, voc["levels"], feats, 2)
    want_v, want_fv = {}, {}
    for i in range(len(feats)):
        w = voc["weight"][wleaf[i]]
        if w > 0:
            want_v[int(voc["word_id"][wleaf[i]])] = want_v.get(int(voc["word_id"][wleaf[i]]), 0.0) + w
            want_fv.setdefault(int(wnid[i]), []).append(i)
    s = sum(abs(want_v[k]) for k in sorted(want_v))
    assert bow == {k: v / s for k, v in want_v.items()}
    assert nodes.tolist() == sorted(want_fv) and idx.tolist() == [i for k in sorted(want_fv) for i in want_fv[k]]
    assert len(nodes) > 5 and abs(sum(bow.values()) - 1.0) < 1e-9
    walk0, _ = V.walk(np.zeros((0, 32), np.uint8))
    assert len(walk0) == 0


def test_matcher_error_conventions():
    import ctypes as C
    from visual_sgraphs_b200 import _lib
    from visual_sgraphs_b200._lib import ptr
    from visual_sgraphs_b200.matcher import ORBmatcher
    L = _lib.load()
    m = ORBmatcher()
    q = np.zeros((4, 32), np.uint8)
    out = np.zeros((4, 2), np.int32)
    assert L.vsg_knn2(m._h, ptr(q), -1, ptr(q), 4, 0, ptr(out), ptr(out)) == _lib.VSG_ERR_INVALID
    assert L.vsg_knn2(None, ptr(q), 4, ptr(q), 4, 0, ptr(out), ptr(out)) == _lib.VSG_ERR_INVALID
    idx, dist = m.knn2(q, np.zeros((0, 32), np.uint8))                     # empty train set: no neighbours
    assert (idx == -1).all() and (dist == np.iinfo(np.int32).max).all()
    bad_ptr = np.array([0, 3, 2], np.int32)                                # decreasing CSR offsets
    assert L.vsg_distinctive_descriptors(m._h, ptr(q), ptr(bad_ptr), 2, ptr(out)) == _lib.VSG_ERR_INVALID
    assert L.vsg_matcher_create(99, C.byref(C.c_void_p())) == _lib.VSG_ERR_CUDA
    # a vocabulary whose child lists do not cover every node exactly once is rejected
    assert L.vsg_vocabulary_create(m._h, 3, ptr(np.array([0, 1, 1, 1], np.int32)), ptr(np.array([1], np.int32)),
                                   ptr(np.zeros((3, 32), np.uint8)), 2, C.byref(C.c_void_p())) == _lib.VSG_ERR_INVALID


def test_frame_create_rejects_views_the_kernels_cannot_index():
    """vsg_frame_create rejects a view whose level tables the searches would read out of bounds: more than kMaxLevels (16)
    levels, no level while there are keypoints, a keypoint octave outside [0, n_levels).  A valid frame created right after
    each rejected one still searches correctly."""
    import ctypes as C
    from visual_sgraphs_b200 import _lib
    from visual_sgraphs_b200._lib import KEYPOINT_DTYPE
    from visual_sgraphs_b200.frame import FrameData
    from visual_sgraphs_b200.matcher import ORBmatcher
    L = _lib.load()
    m = ORBmatcher()
    rng = np.random.default_rng(3)
    keys = np.zeros(200, KEYPOINT_DTYPE)
    keys["x"], keys["y"] = rng.uniform(0, 640, 200), rng.uniform(0, 480, 200)
    keys["octave"] = rng.integers(0, 8, 200)
    desc = rng.integers(0, 256, (200, 32), dtype=np.uint8)
    scale8 = FrameData(keys, desc).scale_factors
    scale16 = np.float32(1.1) ** np.arange(16, dtype=np.float32)

    def with_octave(i, o):
        k = keys.copy()
        k["octave"][i] = o
        return k

    def rejected(data, what):
        h = C.c_void_p()
        assert L.vsg_frame_create(m._h, C.byref(data.view), C.byref(h)) == _lib.VSG_ERR_INVALID, what
        assert not h.value, what
        assert b"vsg_frame_create" in L.vsg_last_error(), what

    valid = FrameData(keys, desc)
    qx, qy = keys["x"][:50].copy(), keys["y"][:50].copy()
    qr = np.full(50, 30, np.float32)
    lo, hi = np.full(50, -1, np.int32), np.full(50, -1, np.int32)
    want = m.area_search(m.frame(valid), qx, qy, qr, lo, hi, desc[:50])
    assert len(want[1]) > 50
    cases = [
        (FrameData(keys, desc, scale_factors=np.concatenate([scale16, [np.float32(5.0)]])), "17 levels"),
        (FrameData(keys, desc, scale_factors=np.zeros(0, np.float32)), "no level, 200 keypoints"),
        (FrameData(with_octave(17, -1), desc), "octave -1"),
        (FrameData(with_octave(199, 8), desc, scale_factors=scale8), "octave 8 of 8 levels"),
        (FrameData(with_octave(0, 16), desc, scale_factors=scale16), "octave 16 of 16 levels"),
    ]
    for data, what in cases:
        rejected(data, what)
        got = m.area_search(m.frame(valid), qx, qy, qr, lo, hi, desc[:50])
        for g, w in zip(got, want):
            assert np.array_equal(g, w), what
    # the limits themselves are accepted: 16 levels with a keypoint on the last one, and an empty view without levels
    m.frame(FrameData(with_octave(0, 15), desc, scale_factors=scale16)).close()
    m.frame(FrameData(np.zeros(0, KEYPOINT_DTYPE), np.zeros((0, 32), np.uint8), scale_factors=np.zeros(0, np.float32))).close()


def test_knn2_full_size_properties():
    """BASELINE config 5 at its full size (100k x 1M descriptors, device-resident): size-independent properties —
    sampled queries against a numpy brute force over the whole train set, planted exact and near duplicates found at
    the right indices, the answer for a query equal to the answer for the same query placed elsewhere in the batch,
    and the train set split into two shards + merge equal to the one-shot result."""
    torch = pytest.importorskip("torch")
    m = _matcher()
    nq, nt = 100_000, 1_000_000
    g = torch.Generator(device="cuda").manual_seed(11)
    q = torch.randint(0, 256, (nq, 32), dtype=torch.uint8, device="cuda", generator=g)
    t = torch.randint(0, 256, (nt, 32), dtype=torch.uint8, device="cuda", generator=g)
    t[999_999] = t[123]                       # exact duplicates across the two halves: the lower index must come first
    q[5] = t[123]
    q[77_777] = t[654_321] ^ torch.tensor([1] + [0] * 31, dtype=torch.uint8, device="cuda")   # one bit away
    q[99_999] = q[42]                         # the same query twice
    idx = torch.zeros((nq, 2), dtype=torch.int32, device="cuda")
    dist = torch.zeros((nq, 2), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    m.knn2_dev(q, t, idx, dist)
    m.sync()
    idx_h, dist_h = idx.cpu().numpy(), dist.cpu().numpy()
    assert tuple(idx_h[5]) == (123, 999_999) and tuple(dist_h[5]) == (0, 0)
    assert idx_h[77_777, 0] == 654_321 and dist_h[77_777, 0] == 1
    assert np.array_equal(idx_h[99_999], idx_h[42]) and np.array_equal(dist_h[99_999], dist_h[42])
    assert (dist_h[:, 0] <= dist_h[:, 1]).all() and (idx_h >= 0).all() and (idx_h < nt).all()
    t_h = t.cpu().numpy()
    sample = np.array([0, 5, 42, 31_337, 77_777, 99_999])
    qs = q[torch.from_numpy(sample).cuda()].cpu().numpy()
    for s, qq in zip(sample, qs):
        d = POP[np.bitwise_xor(t_h, qq[None, :])].sum(1)
        order = np.argsort(d.astype(np.int64) * (1 << 32) + np.arange(nt), kind="stable")[:2]
        assert np.array_equal(idx_h[s], order) and np.array_equal(dist_h[s], d[order]), s
    # two shards + merge == one shot
    half = nt // 2
    parts_i = torch.zeros((2, nq, 2), dtype=torch.int32, device="cuda")
    parts_d = torch.zeros((2, nq, 2), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    m.knn2_dev(q, t[:half].contiguous(), parts_i[0], parts_d[0], 0)
    m.knn2_dev(q, t[half:].contiguous(), parts_i[1], parts_d[1], half)
    mi = torch.zeros((nq, 2), dtype=torch.int32, device="cuda")
    md = torch.zeros((nq, 2), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    m.knn2_merge_dev(parts_i, parts_d, mi, md)
    m.sync()
    assert torch.equal(mi, idx) and torch.equal(md, dist)


def test_sharded_entry_points_on_a_single_rank_communicator(oracle):
    """vsg_comm_* / vsg_knn2_sharded / vsg_search_by_projection_map_sharded with a one-rank NCCL communicator (the
    pytest box has one GPU): the plumbing behind the C ABI — dlopen of NCCL, communicator, all-gather, merge, the replay
    from the claim token — must reproduce the single-GPU calls.  The N > 1 runs are bench.py's `matching_sharded`
    block (torchrun) and tools/multi_gpu_check.py."""
    import torch
    from tests import match_scenarios as sc
    from visual_sgraphs_b200.comm import Comm
    from visual_sgraphs_b200.matcher import ORBmatcher
    assert Comm.nccl_version() >= 21000
    comm = Comm(Comm.unique_id(), 1, 0, 0)
    m = ORBmatcher(nnratio=0.8, device=0)
    q, t = synth_query_train(9, 300, 20000)
    qd, td = torch.from_numpy(q).cuda(), torch.from_numpy(t).cuda()
    i0, d0 = (torch.zeros((300, 2), dtype=torch.int32, device="cuda") for _ in range(2))
    i1, d1 = (torch.zeros((300, 2), dtype=torch.int32, device="cuda") for _ in range(2))
    m.knn2_dev(qd, td, i0, d0)
    m.knn2_sharded(comm, qd, td, 0, i1, d1)
    m.sync()
    assert torch.equal(i0, i1) and torch.equal(d0, d1)
    ka, da, kb, db = sc.two_frames(oracle)
    fd = sc.frame_data(ka, da, stereo_seed=5)
    kb2, db2 = np.concatenate([kb] * 6), np.concatenate([db] * 6)
    pts, desc, occ = sc.track_points(fd, kb2, db2, (9, 5), 21, True)
    frame = m.frame(fd)
    want = m.SearchByProjectionMap(frame, occ, pts, desc, 3.0)
    got = m.SearchByProjectionMapSharded(comm, frame, occ, 0, pts, desc, 3.0)
    assert got[0] == want[0] and np.array_equal(got[1], want[1]) and want[0] > 100
    onm, oassign = oracle.search_by_projection_map(fd.view, occ, pts, desc, 3.0, False, 50.0, float(np.float32(0.8)))
    assert got[0] == onm and np.array_equal(got[1], oassign)
    comm.close()
    m.close()


@pytest.mark.parametrize("nq,nt", [(1, 2), (5, 130), (256, 4096), (300, 5000), (1030, 20000), (777, 128 * 37 + 5), (2000, 3)])
def test_knn2_tensor_core_path_matches_bruteforce(nq, nt, monkeypatch):
    """The tcgen05.mma.kind::i8 formulation (csrc/knn_tc.cu: descriptors expanded to +-1 bytes, dot = 256 - 2 * Hamming,
    top-2 epilogue out of tensor memory) forced on at small shapes (VSG_KNN_TC=2): distances AND indices must equal the
    brute-force (distance, index) top-2 — ties to the lower train index, ragged last tiles, rows past nq / nt ignored."""
    monkeypatch.setenv("VSG_KNN_TC", "2")
    q, t = synth_query_train(nq * 13 + nt, nq, nt)
    if nt >= 8:
        t[3] = t[1]
        t[nt - 1] = t[1]      # a tie in the last (partial) tile
        q[0] = t[1]
    idx, dist = _matcher().knn2(q, t, train_index_offset=1000)
    widx, wdist = knn2_ref(q, t)
    assert np.array_equal(dist, wdist)
    assert np.array_equal(idx, widx + 1000)
    monkeypatch.setenv("VSG_KNN_TC", "0")
    idx0, dist0 = _matcher().knn2(q, t, train_index_offset=1000)
    assert np.array_equal(idx0, idx) and np.array_equal(dist0, dist)
