"""CPU-only, world_size 2 over gloo: the N>1 host logic of the train-sharded kNN-2 (shard bounds, global index
offsets, all-gather, (distance, index) merge) gives exactly the single-process brute-force answer."""
import os
import socket

import numpy as np
import pytest

torch = pytest.importorskip("torch")
import torch.distributed as dist  # noqa: E402
import torch.multiprocessing as mp  # noqa: E402

from visual_sgraphs_b200 import sharded  # noqa: E402
from visual_sgraphs_b200.synth import synth_query_train  # noqa: E402

POP = np.array([bin(i).count("1") for i in range(256)], np.int32)


def knn2_numpy(q, t, offset=0):
    nq = q.shape[0]
    idx = np.full((nq, 2), -1, np.int32)
    d = np.full((nq, 2), np.iinfo(np.int32).max, np.int32)
    if t.shape[0]:
        dm = POP[np.bitwise_xor(q[:, None, :], t[None, :, :])].sum(-1).astype(np.int64)
        key = dm * (1 << 32) + np.arange(t.shape[0])[None, :]
        order = np.argsort(key, axis=1, kind="stable")[:, :2]
        k = order.shape[1]
        idx[:, :k] = order + offset
        d[:, :k] = np.take_along_axis(dm, order, 1)
    return idx, d


def _worker(rank, world, port, nq, nt, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    q, t = synth_query_train(5, nq, nt)
    if nt > 7:
        t[7] = t[nt - 3]                   # a tie across shards must resolve to the lower global index
        q[0] = t[7]
    b, e = sharded.shard_bounds(nt, world)[rank]

    def local(qq, tt, off):
        i, d = knn2_numpy(qq, tt, off)
        return torch.from_numpy(i), torch.from_numpy(d)

    def merge(ip, dp):
        return sharded.merge_top2_numpy(ip.numpy(), dp.numpy())

    idx, d = sharded.knn2_sharded(dist, q, t[b:e], b, local, merge, lambda shape: torch.zeros(shape, dtype=torch.int32))
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), idx=idx, dist=d)
    dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_shard_bounds():
    assert sharded.shard_bounds(10, 4) == [(0, 3), (3, 6), (6, 8), (8, 10)]
    assert sharded.shard_bounds(2, 4) == [(0, 1), (1, 2), (2, 2), (2, 2)]
    assert sharded.frame_shard(1000, 7, 8) == (875, 1000)


@pytest.mark.parametrize("nt", [301, 1])
def test_train_sharded_knn2_over_gloo(tmp_path, nt):
    world, nq = 2, 64
    mp.spawn(_worker, args=(world, _free_port(), nq, nt, str(tmp_path)), nprocs=world, join=True)
    q, t = synth_query_train(5, nq, nt)
    if nt > 7:
        t[7] = t[nt - 3]
        q[0] = t[7]
    want_i, want_d = knn2_numpy(q, t)
    for r in range(world):
        got = np.load(str(tmp_path / ("rank%d.npz" % r)))
        assert np.array_equal(got["idx"], want_i)
        assert np.array_equal(got["dist"], want_d)
    if nt > 7:
        assert want_i[0, 0] == 7 and want_i[0, 1] == nt - 3 and want_d[0, 0] == 0 and want_d[0, 1] == 0


# ---- map-point-sharded SearchByProjection (BASELINE config 3) ----
def _proj_scenario(oracle):
    from tests import match_scenarios as sc
    ka, da, kb, db = sc.two_frames(oracle, size=(322, 243), nfeat=400)
    fd = sc.frame_data(ka, da, size=(322, 243), stereo_seed=5)
    reps = 5
    kb2, db2 = np.concatenate([kb] * reps), np.concatenate([db] * reps)
    pts, desc, occ = sc.track_points(fd, kb2, db2, (9, 5), 21, True)
    return fd, pts, desc, occ


def _cpu_candidates(oracle, fd, pts, desc, th):
    """CPU stand-in for vsg_projection_map_candidates built from the oracle's GetFeaturesInArea restatement."""
    f32 = np.float32
    ptr, idx, dist = [0], [], []
    for i, mp in enumerate(pts):
        if mp["in_view"] and not mp["bad"]:
            lvl = int(mp["level"])
            r = f32(2.5) if float(mp["view_cos"]) > 0.998 else f32(4.0)
            if th != 1.0:
                r = f32(r * f32(th))
            win = f32(r * fd.scale_factors[lvl])
            for j in oracle.get_features_in_area(fd.view, float(mp["proj_x"]), float(mp["proj_y"]), float(win), lvl - 1, lvl):
                if fd.u_right is not None and fd.u_right[j] > 0 and abs(f32(mp["proj_xr"] - fd.u_right[j])) > win:
                    continue
                idx.append(j)
                dist.append(oracle.descriptor_distance(desc[i], fd.descriptors[j]))
        ptr.append(len(idx))
    return np.array(ptr, np.int32), np.array(idx, np.int32), np.array(dist, np.int32)


def _proj_worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from oracle import oracle as orc
    from visual_sgraphs_b200.matcher import projection_map_resolve
    fd, pts, desc, occ = _proj_scenario(orc)
    b, e = sharded.shard_bounds(len(pts), world)[rank]
    nm, assign = sharded.search_by_projection_map_sharded(
        dist, len(pts), pts[b:e], lambda: _cpu_candidates(orc, fd, pts[b:e], desc[b:e], 3.0),
        lambda pa, cp, ci, cd: projection_map_resolve(fd, occ, pa, cp, ci, cd, 0.8))
    np.savez(os.path.join(out_dir, "proj%d.npz" % rank), nm=nm, assign=assign)
    dist.destroy_process_group()


def test_map_sharded_search_by_projection_over_gloo(tmp_path, oracle):
    world = 2
    mp.spawn(_proj_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    fd, pts, desc, occ = _proj_scenario(oracle)
    wnm, wassign = oracle.search_by_projection_map(fd.view, occ, pts, desc, 3.0, False, 50.0, float(np.float32(0.8)))
    assert wnm > 50
    for r in range(world):
        got = np.load(str(tmp_path / ("proj%d.npz" % r)))
        assert int(got["nm"]) == wnm and np.array_equal(got["assign"], wassign)


# ---- the token-ring form the C ABI implements with NCCL (vsg_search_by_projection_map_sharded) ----
def test_shard_by_shard_replay_equals_the_one_call_resolve(oracle):
    """vsg_projection_map_resolve_shard chained over 1, 2, 3 and 7 contiguous shards (claim state carried from shard to
    shard, later shards overwriting slots) == vsg_projection_map_resolve on the whole map == the oracle's one-call method."""
    from visual_sgraphs_b200.matcher import projection_map_resolve, projection_map_resolve_shard
    fd, pts, desc, occ = _proj_scenario(oracle)
    wnm, wassign = oracle.search_by_projection_map(fd.view, occ, pts, desc, 3.0, False, 50.0, float(np.float32(0.8)))
    cp, ci, cd = _cpu_candidates(oracle, fd, pts, desc, 3.0)
    nm1, a1 = projection_map_resolve(fd, occ, pts, cp, ci, cd, 0.8)
    assert nm1 == wnm and np.array_equal(a1, wassign)
    for world in (1, 2, 3, 7):
        blocked = np.ascontiguousarray(occ, np.uint8).copy()
        assign = np.full(fd.n, -1, np.int32)
        total = 0
        for b, e in sharded.shard_bounds(len(pts), world):
            lp = (cp[b:e + 1] - cp[b]).astype(np.int32)
            total += projection_map_resolve_shard(fd, blocked, assign, b, pts[b:e], lp, ci[cp[b]:cp[e]], cd[cp[b]:cp[e]], 0.8)
        assert total == wnm and np.array_equal(assign, wassign), world


def test_shard_replay_rejects_a_bad_index_before_writing(oracle):
    """A candidate index out of range in the last map point's list: vsg_projection_map_resolve_shard fails and leaves the
    claim state and the assignments untouched, although earlier map points of the shard would have matched."""
    from visual_sgraphs_b200 import _lib
    from visual_sgraphs_b200.matcher import projection_map_resolve_shard
    fd, pts, desc, occ = _proj_scenario(oracle)
    cp, ci, cd = _cpu_candidates(oracle, fd, pts, desc, 3.0)
    assert projection_map_resolve_shard(fd, np.ascontiguousarray(occ, np.uint8).copy(), np.full(fd.n, -1, np.int32), 0,
                                        pts[:-1], cp[:-1], ci, cd, 0.8) > 0
    ci, cd, cp = np.append(ci, fd.n).astype(np.int32), np.append(cd, 0).astype(np.int32), cp.copy()
    cp[-1] += 1
    blocked = np.ascontiguousarray(occ, np.uint8).copy()
    assign = np.full(fd.n, -1, np.int32)
    with pytest.raises(_lib.VsgError, match="candidate index out of range"):
        projection_map_resolve_shard(fd, blocked, assign, 0, pts, cp, ci, cd, 0.8)
    assert np.array_equal(blocked, np.ascontiguousarray(occ, np.uint8)) and (assign == -1).all()


def _ring_worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from oracle import oracle as orc
    from visual_sgraphs_b200.matcher import projection_map_resolve_shard
    fd, pts, desc, occ = _proj_scenario(orc)
    b, e = sharded.shard_bounds(len(pts), world)[rank]
    cp, ci, cd = _cpu_candidates(orc, fd, pts[b:e], desc[b:e], 3.0)
    nm, assign = sharded.search_by_projection_map_token_ring(
        dist, fd.n, occ, b, lambda blocked, a: projection_map_resolve_shard(fd, blocked, a, b, pts[b:e], cp, ci, cd, 0.8))
    np.savez(os.path.join(out_dir, "ring%d.npz" % rank), nm=nm, assign=assign)
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_token_ring_search_by_projection_over_gloo(tmp_path, oracle, world):
    mp.spawn(_ring_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    fd, pts, desc, occ = _proj_scenario(oracle)
    wnm, wassign = oracle.search_by_projection_map(fd.view, occ, pts, desc, 3.0, False, 50.0, float(np.float32(0.8)))
    for r in range(world):
        got = np.load(str(tmp_path / ("ring%d.npz" % r)))
        assert int(got["nm"]) == wnm and np.array_equal(got["assign"], wassign)
