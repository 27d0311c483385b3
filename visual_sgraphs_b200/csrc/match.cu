// match.cu — 256-bit Hamming matching kernels behind the matcher half of the C ABI.
//
// Reference (snt-arg/visual_sgraphs):
//   ORBmatcher::DescriptorDistance      orb_slam3/src/ORBmatcher.cc:2047-2063   (8 x 32-bit XOR + popcount)
//   best / second-best candidate scans  :77-120 (SearchByProjection), :670-695 (SearchForInitialization), ...
//   cv::BFMatcher(NORM_HAMMING).knnMatch(q, t, 2)   Frame.cc:1200  (ties: lower train index first, SURVEY A7)
//
// Integer work on the POPC pipe; tensor cores are deliberately not used (north star).  Each distance
// is 8 LOP3 (xor) + 8 POPC + 4 IADD3; the top-2 state is a pair of packed (distance << 23 | index)
// keys updated with integer min/max, which orders candidates lexicographically by (distance, index) —
// the same order a strict '<' scan over increasing indices produces.
#include <algorithm>
#include <climits>

#include "vsg_internal.cuh"
#include "comm_internal.h"

namespace vsg {

vsg_status matcher_ensure(vsg_matcher *m, DevSlot slot, size_t bytes) {
    if (m->cap[slot] >= bytes) return VSG_OK;
    if (m->buf[slot]) cudaFree(m->buf[slot]);
    m->buf[slot] = nullptr;
    m->cap[slot] = 0;
    const size_t want = bytes + bytes / 4 + 256;
    CK(cudaMalloc(&m->buf[slot], want));
    m->cap[slot] = want;
    return VSG_OK;
}
vsg_status matcher_ensure_host(vsg_matcher *m, HostSlot slot, size_t bytes) {
    if (m->hcap[slot] >= bytes) return VSG_OK;
    if (m->hbuf[slot]) cudaFreeHost(m->hbuf[slot]);
    m->hbuf[slot] = nullptr;
    m->hcap[slot] = 0;
    const size_t want = bytes + bytes / 4 + 256;
    CK(cudaMallocHost(&m->hbuf[slot], want));
    m->hcap[slot] = want;
    return VSG_OK;
}

__device__ __forceinline__ int hamming256(const uint4 &a0, const uint4 &a1, const uint4 &b0, const uint4 &b1) {
    return __popc(a0.x ^ b0.x) + __popc(a0.y ^ b0.y) + __popc(a0.z ^ b0.z) + __popc(a0.w ^ b0.w) +
           __popc(a1.x ^ b1.x) + __popc(a1.y ^ b1.y) + __popc(a1.z ^ b1.z) + __popc(a1.w ^ b1.w);
}

// ------------------------------------------------------------------------------------------------
// pairwise distances
// ------------------------------------------------------------------------------------------------
__global__ void pair_distance_kernel(const uint4 *__restrict__ a, const uint4 *__restrict__ b, int n,
                                     int *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = hamming256(__ldg(a + 2 * i), __ldg(a + 2 * i + 1), __ldg(b + 2 * i), __ldg(b + 2 * i + 1));
}

// ------------------------------------------------------------------------------------------------
// brute-force kNN (k = 2).  grid (query tiles, train chunks), 256 threads, kQ queries per thread.
// Train rows are staged through shared memory in tiles of 256 rows; every thread reads the same row
// at the same time (shared-memory broadcast).  Partial top-2 per (query, chunk) goes to scratch and
// is merged by knn2_merge_kernel in chunk order.
// ------------------------------------------------------------------------------------------------
constexpr int kKnnThreads = 256;
constexpr int kKnnQ = 4;          // queries per thread
constexpr int kKnnTile = 256;     // train rows per shared-memory tile
constexpr unsigned kKeyIdxBits = 23;
constexpr unsigned kKeyEmpty = 0xFFFFFFFFu;

__global__ void __launch_bounds__(kKnnThreads) knn2_kernel(const uint4 *__restrict__ query, int nq,
                                                          const uint4 *__restrict__ train, int nt, int chunk_rows,
                                                          unsigned *__restrict__ part_keys /* [chunks][nq][2] */) {
    __shared__ uint4 tile[2][kKnnTile * 2];
    const int tid = threadIdx.x;
    const int q0 = (blockIdx.x * kKnnThreads + tid) * kKnnQ;
    const int t_begin = blockIdx.y * chunk_rows;
    const int t_end = min(t_begin + chunk_rows, nt);

    uint4 qa[kKnnQ], qb[kKnnQ];
    unsigned k1[kKnnQ], k2[kKnnQ];
#pragma unroll
    for (int j = 0; j < kKnnQ; ++j) {
        const int q = min(q0 + j, nq - 1);
        qa[j] = __ldg(query + 2 * q);
        qb[j] = __ldg(query + 2 * q + 1);
        k1[j] = kKeyEmpty;
        k2[j] = kKeyEmpty;
    }
    const int ntiles = (t_end - t_begin + kKnnTile - 1) / kKnnTile;
    auto load_tile = [&](int t, int buf) {
        const int row = t_begin + t * kKnnTile + tid;
        uint4 lo = make_uint4(0, 0, 0, 0), hi = lo;
        if (row < t_end) { lo = __ldg(train + 2 * row); hi = __ldg(train + 2 * row + 1); }
        tile[buf][2 * tid] = lo;
        tile[buf][2 * tid + 1] = hi;
    };
    if (ntiles > 0) load_tile(0, 0);
    __syncthreads();
    for (int t = 0; t < ntiles; ++t) {
        const int buf = t & 1;
        if (t + 1 < ntiles) load_tile(t + 1, buf ^ 1);
        const int rows = min(kKnnTile, t_end - t_begin - t * kKnnTile);
        const unsigned local0 = (unsigned)(t * kKnnTile);
#pragma unroll 4
        for (int r = 0; r < rows; ++r) {
            const uint4 ta = tile[buf][2 * r], tb = tile[buf][2 * r + 1];
#pragma unroll
            for (int j = 0; j < kKnnQ; ++j) {
                const unsigned d = (unsigned)hamming256(qa[j], qb[j], ta, tb);
                const unsigned key = (d << kKeyIdxBits) | (local0 + r);
                k2[j] = min(k2[j], max(k1[j], key));
                k1[j] = min(k1[j], key);
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int j = 0; j < kKnnQ; ++j) {
        const int q = q0 + j;
        if (q < nq) {
            unsigned *o = part_keys + ((size_t)blockIdx.y * nq + q) * 2;
            o[0] = k1[j];
            o[1] = k2[j];
        }
    }
}

// Merge per-chunk partial keys (chunk-local indices) into global (idx, dist) pairs.
__global__ void knn2_merge_kernel(const unsigned *__restrict__ part_keys, int nchunks, int nq, int chunk_rows,
                                  int index_offset, int *__restrict__ out_idx, int *__restrict__ out_dist) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    unsigned long long b1 = ~0ull, b2 = ~0ull;  // (dist << 32 | global idx)
    for (int c = 0; c < nchunks; ++c) {
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            const unsigned k = part_keys[((size_t)c * nq + q) * 2 + s];
            if (k == kKeyEmpty) continue;
            const unsigned long long key = ((unsigned long long)(k >> kKeyIdxBits) << 32) |
                                           (unsigned long long)((k & ((1u << kKeyIdxBits) - 1)) + (unsigned)c * chunk_rows);
            if (key < b1) { b2 = b1; b1 = key; }
            else if (key < b2) b2 = key;
        }
    }
    out_idx[2 * q] = b1 == ~0ull ? -1 : (int)(b1 & 0xFFFFFFFFull) + index_offset;
    out_dist[2 * q] = b1 == ~0ull ? INT_MAX : (int)(b1 >> 32);
    out_idx[2 * q + 1] = b2 == ~0ull ? -1 : (int)(b2 & 0xFFFFFFFFull) + index_offset;
    out_dist[2 * q + 1] = b2 == ~0ull ? INT_MAX : (int)(b2 >> 32);
}

// Merge `nparts` already-global top-2 lists (after an all-gather over train shards).
__global__ void knn2_merge_parts_kernel(const int *__restrict__ idx_parts, const int *__restrict__ dist_parts,
                                        int nparts, int nq, int *__restrict__ out_idx, int *__restrict__ out_dist) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    unsigned long long b1 = ~0ull, b2 = ~0ull;
    for (int p = 0; p < nparts; ++p) {
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            const int idx = idx_parts[((size_t)p * nq + q) * 2 + s];
            if (idx < 0) continue;
            const unsigned long long key =
                ((unsigned long long)(unsigned)dist_parts[((size_t)p * nq + q) * 2 + s] << 32) | (unsigned)idx;
            if (key < b1) { b2 = b1; b1 = key; }
            else if (key < b2) b2 = key;
        }
    }
    out_idx[2 * q] = b1 == ~0ull ? -1 : (int)(b1 & 0xFFFFFFFFull);
    out_dist[2 * q] = b1 == ~0ull ? INT_MAX : (int)(b1 >> 32);
    out_idx[2 * q + 1] = b2 == ~0ull ? -1 : (int)(b2 & 0xFFFFFFFFull);
    out_dist[2 * q + 1] = b2 == ~0ull ? INT_MAX : (int)(b2 >> 32);
}

// ------------------------------------------------------------------------------------------------
// candidate-list scan: one thread per query walks its CSR candidate list in order with strict '<'
// updates (ORBmatcher.cc:84-120 and the same idiom in every Search* method).
// ------------------------------------------------------------------------------------------------
__global__ void window_match_kernel(const uint4 *__restrict__ query, int nq, const uint4 *__restrict__ train,
                                    const int *__restrict__ cand_ptr, const int *__restrict__ cand,
                                    const uint8_t *__restrict__ skip, const int *__restrict__ train_level,
                                    int init_dist, int *__restrict__ best_idx, int *__restrict__ best_dist,
                                    int *__restrict__ second_dist, int *__restrict__ best_level,
                                    int *__restrict__ second_level) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const uint4 qa = __ldg(query + 2 * q), qb = __ldg(query + 2 * q + 1);
    int bd = init_dist, bd2 = init_dist, bi = -1, bl = -1, bl2 = -1;
    const int e = cand_ptr[q + 1];
    for (int c = cand_ptr[q]; c < e; ++c) {
        const int j = cand[c];
        const int d = hamming256(qa, qb, __ldg(train + 2 * j), __ldg(train + 2 * j + 1));
        if (skip && skip[j]) continue;
        const int lvl = train_level ? train_level[j] : -1;
        if (d < bd) { bd2 = bd; bd = d; bl2 = bl; bl = lvl; bi = j; }
        else if (d < bd2) { bl2 = lvl; bd2 = d; }
    }
    if (best_idx) best_idx[q] = bi;
    if (best_dist) best_dist[q] = bd;
    if (second_dist) second_dist[q] = bd2;
    if (best_level) best_level[q] = bl;
    if (second_level) second_level[q] = bl2;
}

// ------------------------------------------------------------------------------------------------
// BoW in-node distances: one thread per (segment, candidate) pair of every merge walk of a call.  Segment s = (query
// descriptor row, first candidate in the uploaded FeatureVector idx arrays, the candidate side's first descriptor row,
// first output slot); the segments are sorted by output slot and end with a sentinel whose slot is npairs.  A thread
// finds its segment by binary search over the slots and writes its distance in walk order (0..256 fits 16 bits).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) bow_dists_multi_kernel(const int4 *__restrict__ segs, int nseg, const int *__restrict__ idx,
                                                              const uint4 *__restrict__ desc, int npairs,
                                                              unsigned short *__restrict__ out) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npairs) return;
    int lo = 0, hi = nseg - 1;                           // last segment whose first slot is <= p
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(&segs[mid].w) <= p) lo = mid;
        else hi = mid - 1;
    }
    const int4 s = __ldg(segs + lo);
    const int j = s.z + __ldg(idx + s.y + (p - s.w));
    out[p] = (unsigned short)hamming256(__ldg(desc + 2 * s.x), __ldg(desc + 2 * s.x + 1), __ldg(desc + 2 * j), __ldg(desc + 2 * j + 1));
}

void launch_bow_dists(vsg_matcher *m, const int4 *segs_dev, int nseg, const int *idx_dev, const uint8_t *desc_dev, int npairs,
                      uint16_t *out_dev) {
    if (npairs <= 0) return;
    bow_dists_multi_kernel<<<(npairs + 255) / 256, 256, 0, m->stream>>>(segs_dev, nseg, idx_dev, (const uint4 *)desc_dev, npairs,
                                                                        out_dev);
    count_launch();
}

// ------------------------------------------------------------------------------------------------
// SearchForTriangulation's per-pair test (ORBmatcher.cc:998-1077 with Pinhole::epipolarConstrain, Pinhole.cpp:126-140): one
// warp per segment, lanes stride over the candidates.  The reference keeps bestDist starting at TH_LOW and accepts on
// `d <= bestDist`, and no gate reads bestDist, so it ends with the minimum distance among the passing candidates, the last
// one in scan order on ties: a warp minimum over (d << 32 | ~position).  The float arithmetic is spelled out with _rn
// intrinsics (no contraction whatever --fmad says, IEEE division) and the chi-square gate compares in double, as the
// reference's `dsqr < 3.84 * sigma2` does.
// ------------------------------------------------------------------------------------------------
constexpr int kTriWarps = 8;

__global__ void __launch_bounds__(kTriWarps * 32) triangulation_best_kernel(const TriSeg *__restrict__ segs, int nseg,
                                                                            const TriTarget *__restrict__ targets,
                                                                            const int *__restrict__ idx, const uint4 *__restrict__ desc,
                                                                            const TriKey *__restrict__ keys,
                                                                            const float2 *__restrict__ lvl, int only_stereo,
                                                                            int coarse, int *__restrict__ out) {
    const int s = blockIdx.x * kTriWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (s >= nseg) return;                                                    // whole warps only
    const TriSeg sg = segs[s];
    const TriTarget &tg = targets[sg.target];
    const uint4 qa = __ldg(desc + 2 * sg.q_row), qb = __ldg(desc + 2 * sg.q_row + 1);
    const float ep0 = __ldg(&tg.ep[0]), ep1 = __ldg(&tg.ep[1]);
    const int desc0 = __ldg(&tg.desc0), key0 = __ldg(&tg.key0), lvl0 = __ldg(&tg.lvl0);
    float a = 0.f, b = 0.f, c = 0.f;                                          // Pinhole.cpp:126-128
    if (!coarse) {
        const float *f = tg.f12;
        a = __fadd_rn(__fadd_rn(__fmul_rn(sg.x1, __ldg(f + 0)), __fmul_rn(sg.y1, __ldg(f + 3))), __ldg(f + 6));
        b = __fadd_rn(__fadd_rn(__fmul_rn(sg.x1, __ldg(f + 1)), __fmul_rn(sg.y1, __ldg(f + 4))), __ldg(f + 7));
        c = __fadd_rn(__fadd_rn(__fmul_rn(sg.x1, __ldg(f + 2)), __fmul_rn(sg.y1, __ldg(f + 5))), __ldg(f + 8));
    }
    unsigned long long best = ~0ull;
    for (int p = lane; p < sg.ncand; p += 32) {
        const int i2 = __ldg(idx + sg.cand + p);
        const int4 kr = __ldg((const int4 *)(keys + key0 + i2));
        const float x2 = __int_as_float(kr.x), y2 = __int_as_float(kr.y);
        if (kr.w & kTriHasMp) continue;                                       // :1001 (vbMatched2 is never set)
        const bool stereo2 = kr.w & kTriStereo;
        if (only_stereo && !stereo2) continue;                                // :1008
        const int d = hamming256(qa, qb, __ldg(desc + 2 * (desc0 + i2)), __ldg(desc + 2 * (desc0 + i2) + 1));
        if (d > 50) continue;                                                 // :1014, TH_LOW
        const float2 lv = __ldg(lvl + lvl0 + kr.z);
        if (!sg.stereo1 && !stereo2) {                                        // :1023-1031
            const float ex = __fsub_rn(ep0, x2), ey = __fsub_rn(ep1, y2);
            if (__fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey)) < __fmul_rn(100.f, lv.x)) continue;
        }
        if (!coarse) {                                                        // Pinhole.cpp:130-140
            const float num = __fadd_rn(__fadd_rn(__fmul_rn(a, x2), __fmul_rn(b, y2)), c);
            const float den = __fadd_rn(__fmul_rn(a, a), __fmul_rn(b, b));
            if (den == 0.f) continue;
            const float dsqr = __fdiv_rn(__fmul_rn(num, num), den);
            if (!((double)dsqr < __dmul_rn(3.84, (double)lv.y))) continue;
        }
        best = min(best, ((unsigned long long)d << 32) | (unsigned)~p);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(0xffffffffu, best, o));
    if (lane == 0) out[s] = best == ~0ull ? -1 : __ldg(idx + sg.cand + (int)~(unsigned)best);
}

void launch_triangulation_best(vsg_matcher *m, const TriSeg *segs_dev, int nseg, const TriTarget *targets_dev, const int *idx_dev,
                               const uint8_t *desc_dev, const TriKey *keys_dev, const float2 *lvl_dev, int only_stereo, int coarse,
                               int *out_dev) {
    if (nseg <= 0) return;
    triangulation_best_kernel<<<(nseg + kTriWarps - 1) / kTriWarps, kTriWarps * 32, 0, m->stream>>>(
        segs_dev, nseg, targets_dev, idx_dev, (const uint4 *)desc_dev, keys_dev, lvl_dev, only_stereo, coarse, out_dev);
    count_launch();
}

static void knn2_plan(const vsg_matcher *m, int nq, int nt, int *qtiles, int *nchunks, int *chunk_rows) {
    *qtiles = (nq + kKnnThreads * kKnnQ - 1) / (kKnnThreads * kKnnQ);
    // enough CTAs for ~4 waves over the SMs, chunks a multiple of the tile size and below the key's index range
    int want = std::max(1, (m->sm_count * 4 + *qtiles - 1) / *qtiles);
    int rows = (nt + want - 1) / want;
    rows = std::max(kKnnTile, (rows + kKnnTile - 1) / kKnnTile * kKnnTile);
    rows = std::min(rows, 1 << 22);
    *chunk_rows = rows;
    *nchunks = std::max(1, (nt + rows - 1) / rows);
}

vsg_status launch_knn2_merge_parts(vsg_matcher *m, const int32_t *idx_parts, const int32_t *dist_parts, int nparts, int nq,
                                   int32_t *out_idx, int32_t *out_dist) {
    knn2_merge_parts_kernel<<<(nq + 255) / 256, 256, 0, m->stream>>>(idx_parts, dist_parts, nparts, nq, out_idx, out_dist);
    count_launch();
    CK(cudaGetLastError());
    return VSG_OK;
}

static vsg_status knn2_device(vsg_matcher *m, const uint8_t *q_dev, int nq, const uint8_t *t_dev, int nt, int offset,
                              int *idx_dev, int *dist_dev) {
    // large problems: the s8 GEMM formulation on the tensor cores (knn_tc.cu); small ones: the POPC kernel below
    if (knn2_tc_supported(nq, nt)) return knn2_tc_device(m, q_dev, nq, t_dev, nt, offset, idx_dev, dist_dev);
    int qtiles, nchunks, chunk_rows;
    knn2_plan(m, nq, nt, &qtiles, &nchunks, &chunk_rows);
    vsg_status st = matcher_ensure(m, kSlotKnnParts, (size_t)nchunks * nq * 2 * sizeof(unsigned));
    if (st != VSG_OK) return st;
    unsigned *part = (unsigned *)m->buf[kSlotKnnParts];
    if (nt > 0) {
        knn2_kernel<<<dim3(qtiles, nchunks), kKnnThreads, 0, m->stream>>>((const uint4 *)q_dev, nq, (const uint4 *)t_dev, nt,
                                                                          chunk_rows, part);
        count_launch();
    } else {
        nchunks = 0;
    }
    knn2_merge_kernel<<<(nq + 255) / 256, 256, 0, m->stream>>>(part, nchunks, nq, chunk_rows, offset, idx_dev, dist_dev);
    count_launch();
    CK(cudaGetLastError());
    return VSG_OK;
}

}  // namespace vsg

using namespace vsg;

extern "C" {

vsg_status vsg_matcher_create(int device, vsg_matcher **out) {
    if (!out) return VSG_ERR_INVALID;
    if (vsg_device_count() <= device || device < 0) {
        set_error("vsg_matcher_create: CUDA device %d not available (this library has no CPU fallback)", device);
        return VSG_ERR_CUDA;
    }
    vsg_matcher *m = new vsg_matcher();
    m->device = device;
    if (!cuda_ok(cudaSetDevice(device), "cudaSetDevice") ||
        !cuda_ok(cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking), "cudaStreamCreate")) {
        delete m;
        return VSG_ERR_CUDA;
    }
    cudaDeviceGetAttribute(&m->sm_count, cudaDevAttrMultiProcessorCount, device);
    {   // frame uploads use the stream-ordered allocator: keep freed blocks in the pool instead of returning them to the OS
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            unsigned long long keep = 256ull << 20;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        } else {
            cudaGetLastError();
        }
    }
    *out = m;
    return VSG_OK;
}

void vsg_matcher_destroy(vsg_matcher *m) {
    if (!m) return;
    cudaSetDevice(m->device);
    if (m->stream) { cudaStreamSynchronize(m->stream); cudaStreamDestroy(m->stream); }
    for (void *b : m->buf) cudaFree(b);
    for (void *b : m->hbuf) cudaFreeHost(b);
    delete m;
}

void *vsg_matcher_stream(vsg_matcher *m) { return m ? (void *)m->stream : nullptr; }

vsg_status vsg_matcher_sync(vsg_matcher *m) {
    if (!m) return VSG_ERR_INVALID;
    CK(cudaStreamSynchronize(m->stream));
    return VSG_OK;
}

vsg_status vsg_descriptor_distance(vsg_matcher *m, const uint8_t *a, const uint8_t *b, int n, int32_t *out) {
    if (!m || n < 0 || (n > 0 && (!a || !b || !out))) return VSG_ERR_INVALID;
    if (n == 0) return VSG_OK;
    CK(cudaSetDevice(m->device));
    vsg_status st;
    if ((st = matcher_ensure(m, kSlotArg1, (size_t)n * 32)) || (st = matcher_ensure(m, kSlotArg2, (size_t)n * 32)) || (st = matcher_ensure(m, kSlotArg3, (size_t)n * 4))) return st;
    CK(cudaMemcpyAsync(m->buf[kSlotArg1], a, (size_t)n * 32, cudaMemcpyHostToDevice, m->stream));
    CK(cudaMemcpyAsync(m->buf[kSlotArg2], b, (size_t)n * 32, cudaMemcpyHostToDevice, m->stream));
    pair_distance_kernel<<<(n + 255) / 256, 256, 0, m->stream>>>((const uint4 *)m->buf[kSlotArg1], (const uint4 *)m->buf[kSlotArg2], n,
                                                                (int *)m->buf[kSlotArg3]);
    count_launch();
    CK(cudaMemcpyAsync(out, m->buf[kSlotArg3], (size_t)n * 4, cudaMemcpyDeviceToHost, m->stream));
    CK(cudaStreamSynchronize(m->stream));
    return VSG_OK;
}

vsg_status vsg_knn2_dev(vsg_matcher *m, const uint8_t *query_dev, int nq, const uint8_t *train_dev, int nt,
                        int train_index_offset, int32_t *out_idx_dev, int32_t *out_dist_dev) {
    if (!m || nq < 0 || nt < 0 || (nq > 0 && (!query_dev || !out_idx_dev || !out_dist_dev)) || (nt > 0 && !train_dev))
        return VSG_ERR_INVALID;
    if (nq == 0) return VSG_OK;
    CK(cudaSetDevice(m->device));
    return knn2_device(m, query_dev, nq, train_dev, nt, train_index_offset, out_idx_dev, out_dist_dev);
}

vsg_status vsg_knn2(vsg_matcher *m, const uint8_t *query, int nq, const uint8_t *train, int nt, int train_index_offset,
                    int32_t *out_idx, int32_t *out_dist) {
    if (!m || nq < 0 || nt < 0 || (nq > 0 && (!query || !out_idx || !out_dist)) || (nt > 0 && !train)) return VSG_ERR_INVALID;
    if (nq == 0) return VSG_OK;
    CK(cudaSetDevice(m->device));
    vsg_status st;
    if ((st = matcher_ensure(m, kSlotArg1, (size_t)nq * 32)) || (st = matcher_ensure(m, kSlotArg2, (size_t)std::max(nt, 1) * 32)) ||
        (st = matcher_ensure(m, kSlotArg3, (size_t)nq * 8)) || (st = matcher_ensure(m, kSlotArg4, (size_t)nq * 8)))
        return st;
    CK(cudaMemcpyAsync(m->buf[kSlotArg1], query, (size_t)nq * 32, cudaMemcpyHostToDevice, m->stream));
    if (nt) CK(cudaMemcpyAsync(m->buf[kSlotArg2], train, (size_t)nt * 32, cudaMemcpyHostToDevice, m->stream));
    st = knn2_device(m, (const uint8_t *)m->buf[kSlotArg1], nq, (const uint8_t *)m->buf[kSlotArg2], nt, train_index_offset, (int *)m->buf[kSlotArg3],
                     (int *)m->buf[kSlotArg4]);
    if (st != VSG_OK) return st;
    CK(cudaMemcpyAsync(out_idx, m->buf[kSlotArg3], (size_t)nq * 8, cudaMemcpyDeviceToHost, m->stream));
    CK(cudaMemcpyAsync(out_dist, m->buf[kSlotArg4], (size_t)nq * 8, cudaMemcpyDeviceToHost, m->stream));
    CK(cudaStreamSynchronize(m->stream));
    return VSG_OK;
}

vsg_status vsg_knn2_merge_dev(vsg_matcher *m, const int32_t *idx_parts_dev, const int32_t *dist_parts_dev, int nparts,
                              int nq, int32_t *out_idx_dev, int32_t *out_dist_dev) {
    if (!m || nparts < 1 || nq < 0 || !idx_parts_dev || !dist_parts_dev || !out_idx_dev || !out_dist_dev) return VSG_ERR_INVALID;
    if (nq == 0) return VSG_OK;
    CK(cudaSetDevice(m->device));
    knn2_merge_parts_kernel<<<(nq + 255) / 256, 256, 0, m->stream>>>(idx_parts_dev, dist_parts_dev, nparts, nq, out_idx_dev,
                                                                    out_dist_dev);
    count_launch();
    CK(cudaGetLastError());
    return VSG_OK;
}

// Brute-force kNN-2 with the TRAIN set sharded over the ranks of a communicator (BASELINE config 5; SURVEY 8e): every rank
// searches its shard (global train indices through train_index_offset), the per-rank (nq x 2) top-2 lists are exchanged by
// ncclAllGather over NVLink and merged on every rank by (distance, index) — the knnMatch tie rule (Frame.cc:1200), so the
// result equals the single-GPU call on the concatenated train set.  Asynchronous on the matcher's stream.
vsg_status vsg_knn2_sharded(vsg_comm *comm, vsg_matcher *m, const uint8_t *query_dev, int nq, const uint8_t *train_shard_dev,
                            int nt_shard, int train_index_offset, int32_t *out_idx_dev, int32_t *out_dist_dev) {
    if (!comm || !m || nq < 0 || nt_shard < 0 || (nq > 0 && (!query_dev || !out_idx_dev || !out_dist_dev)) ||
        (nt_shard > 0 && !train_shard_dev))
        return VSG_ERR_INVALID;
    if (nq == 0) return VSG_OK;
    CK(cudaSetDevice(m->device));
    const int nranks = comm_size(comm);
    const size_t part = (size_t)nq * 2 * sizeof(int32_t);
    vsg_status st;
    if ((st = matcher_ensure(m, kSlotKnnSharded, 2 * part * (size_t)(nranks + 1)))) return st;
    int32_t *my_idx = (int32_t *)m->buf[kSlotKnnSharded], *my_dist = my_idx + (size_t)nq * 2;
    int32_t *all_idx = my_dist + (size_t)nq * 2, *all_dist = all_idx + (size_t)nq * 2 * nranks;
    if ((st = knn2_device(m, query_dev, nq, train_shard_dev, nt_shard, train_index_offset, my_idx, my_dist)) != VSG_OK) return st;
    if ((st = comm_all_gather(comm, my_idx, all_idx, part, m->stream)) != VSG_OK) return st;
    if ((st = comm_all_gather(comm, my_dist, all_dist, part, m->stream)) != VSG_OK) return st;
    knn2_merge_parts_kernel<<<(nq + 255) / 256, 256, 0, m->stream>>>(all_idx, all_dist, nranks, nq, out_idx_dev, out_dist_dev);
    count_launch();
    CK(cudaGetLastError());
    return VSG_OK;
}

vsg_status vsg_match_window(vsg_matcher *m, const uint8_t *query, int nq, const uint8_t *train, int nt,
                            const int32_t *cand_ptr, const int32_t *cand, const uint8_t *skip,
                            const int32_t *train_level, int init_dist, int32_t *best_idx, int32_t *best_dist,
                            int32_t *second_dist, int32_t *best_level, int32_t *second_level) {
    if (!m || nq < 0 || nt < 0 || (nq > 0 && (!query || !cand_ptr))) return VSG_ERR_INVALID;
    if (nq == 0) return VSG_OK;
    const int ncand = cand_ptr[nq];
    if (ncand < 0 || (ncand > 0 && (!cand || !train))) return VSG_ERR_INVALID;
    CK(cudaSetDevice(m->device));
    vsg_status st;
    if ((st = matcher_ensure(m, kSlotArg1, (size_t)nq * 32)) || (st = matcher_ensure(m, kSlotArg2, (size_t)std::max(nt, 1) * 32)) ||
        (st = matcher_ensure(m, kSlotArg3, (size_t)(nq + 1) * 4)) || (st = matcher_ensure(m, kSlotArg4, (size_t)std::max(ncand, 1) * 4)) ||
        (st = matcher_ensure(m, kSlotArg5, (size_t)std::max(nt, 1) * 5 + 16)) || (st = matcher_ensure(m, kSlotOut, (size_t)nq * 20)))
        return st;
    cudaStream_t s = m->stream;
    CK(cudaMemcpyAsync(m->buf[kSlotArg1], query, (size_t)nq * 32, cudaMemcpyHostToDevice, s));
    if (nt) CK(cudaMemcpyAsync(m->buf[kSlotArg2], train, (size_t)nt * 32, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(m->buf[kSlotArg3], cand_ptr, (size_t)(nq + 1) * 4, cudaMemcpyHostToDevice, s));
    if (ncand) CK(cudaMemcpyAsync(m->buf[kSlotArg4], cand, (size_t)ncand * 4, cudaMemcpyHostToDevice, s));
    int *lvl_dev = (int *)m->buf[kSlotArg5];
    uint8_t *skip_dev = (uint8_t *)m->buf[kSlotArg5] + (size_t)std::max(nt, 1) * 4;
    if (train_level && nt) CK(cudaMemcpyAsync(lvl_dev, train_level, (size_t)nt * 4, cudaMemcpyHostToDevice, s));
    if (skip && nt) CK(cudaMemcpyAsync(skip_dev, skip, (size_t)nt, cudaMemcpyHostToDevice, s));
    int *o = (int *)m->buf[kSlotOut];
    window_match_kernel<<<(nq + 127) / 128, 128, 0, s>>>((const uint4 *)m->buf[kSlotArg1], nq, (const uint4 *)m->buf[kSlotArg2],
                                                        (const int *)m->buf[kSlotArg3], (const int *)m->buf[kSlotArg4],
                                                        skip ? skip_dev : nullptr, train_level ? lvl_dev : nullptr,
                                                        init_dist, o, o + nq, o + 2 * nq, o + 3 * nq, o + 4 * nq);
    count_launch();
    CK(cudaGetLastError());
    int32_t *outs[5] = {best_idx, best_dist, second_dist, best_level, second_level};
    for (int k = 0; k < 5; ++k)
        if (outs[k]) CK(cudaMemcpyAsync(outs[k], o + (size_t)k * nq, (size_t)nq * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return VSG_OK;
}

}  // extern "C"
