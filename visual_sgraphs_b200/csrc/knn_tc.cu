// knn_tc.cu — brute-force Hamming kNN-2 as the dense integer contraction it is, on the 5th-generation tensor cores.
//
// Reference (snt-arg/visual_sgraphs): cv::BFMatcher(NORM_HAMMING).knnMatch(q, t, 2), orb_slam3/src/Frame.cc:1200; the
// distance is ORBmatcher::DescriptorDistance, orb_slam3/src/ORBmatcher.cc:2047-2063 (BASELINE config 5: 100k x 1M).
//
// A 256-bit descriptor expanded to 256 int8 values (+1 for a set bit, -1 for a clear one) turns the Hamming distance into a
// dot product:  dot(a, b) = (#equal bits) - (#different bits) = 256 - 2 * hamming(a, b)  — exact in int32.  The POPC
// formulation (match.cu: knn2_kernel) is bound by the XU pipe at 16 POPC / clk / SM (191 ms for 100k x 1M); the same pairs as
// an s8 GEMM run on tcgen05.mma.kind::i8 with the accumulators in tensor memory.
//
// One persistent CTA per SM, warp-specialised (the canonical sm_100 GEMM shape):
//   warp 0      TMA producer: the item's 256 query rows once (4 boxes of 128 rows x 128 B, SWIZZLE_128B), then the train rows
//               of its segment as a 4-stage ring of 128-row tiles (2 boxes each), mbarrier complete_tx
//   warp 1      MMA issuer (one lane): per train tile 2 (query halves) x 2 (K halves) x 4 tcgen05.mma.cta_group::1.kind::i8 of
//               M128 x N128 x K32 into one of two accumulator stages (2 x 2 x 128 TMEM columns = all 512), tcgen05.commit
//   warps 2..9  epilogue: each thread owns ONE query row (its TMEM lane): tcgen05.ld 32 columns at a time, a max3 tree over
//               the 32 dot products (1/2 instruction per pair), and only if that maximum beats the row's running second-best
//               dot product — about 2 / (pairs seen so far) of the time — the 32 values are scanned for the top-2 update.
//               Columns are visited in increasing train index and updates are strict, so ties keep the lower index: the
//               (distance, index) order of knnMatch.
// Work items = (256-query block, train segment); the per-segment top-2 lists are merged by knn2_merge_parts_kernel (match.cu),
// the same merge the multi-GPU path uses.  Results are bit-identical to knn2_kernel (tests/test_gpu_matcher.py).
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cstdint>
#include <cstdlib>

#include "tma_util.cuh"
#include "vsg_internal.cuh"

namespace vsg {

constexpr int kTcRowsPerItem = 256;     // query rows per work item: two UMMA_M = 128 halves
constexpr int kTcTileN = 128;           // train rows per tile = UMMA_N
constexpr int kTcStages = 4;            // train-tile ring
constexpr int kTcThreads = 32 * 10;     // producer, MMA, 8 epilogue warps
constexpr int kTcBoxBytes = 128 * 128;  // one TMA box: 128 rows x 128 bytes (one SWIZZLE_128B atom wide)
constexpr int kTcSmemA = 4 * kTcBoxBytes;              // [query half][K half]
constexpr int kTcSmemBStage = 2 * kTcBoxBytes;         // [K half]
constexpr int kTcSmemBytes = kTcSmemA + kTcStages * kTcSmemBStage + 256 /* barriers */ + 1024 /* alignment slack */;

__device__ __forceinline__ int max3i(int a, int b, int c) { return max(max(a, b), c); }

// instruction descriptor of kind::i8: D = s32 (bits 4-5 = 2), A and B signed 8-bit (bits 7-9 / 10-12 = 1), both K-major
// (bits 15, 16 = 0), N >> 3 at bit 17, M >> 4 at bit 24
constexpr uint32_t kTcIdesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kTcTileN >> 3) << 17) | ((128u >> 4) << 24);

// descriptor bits -> 256 signed bytes per row: +1 for a set bit, -1 for a clear one (bit i of byte b = element 8 b + i)
__global__ void __launch_bounds__(256) expand_pm1_kernel(const uint32_t *__restrict__ bits, int nrows, int8_t *__restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // one thread per 32-bit word -> 32 output bytes
    if (t >= (int64_t)nrows * 8) return;
    const uint32_t w = __ldg(bits + t);
    uint4 o[2];
    uint32_t *p = reinterpret_cast<uint32_t *>(o);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const uint32_t nib = (w >> (4 * k)) & 0xFu;
        // bytes: bit set -> 0x01, clear -> 0xFF
        uint32_t v = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) v |= (((nib >> b) & 1u) ? 0x01u : 0xFFu) << (8 * b);
        p[k] = v;
    }
    uint4 *dst = reinterpret_cast<uint4 *>(out + t * 32);
    dst[0] = o[0];
    dst[1] = o[1];
}

__global__ void __launch_bounds__(kTcThreads, 1)
knn2_tc_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_t, int nq, int nt, int nitems,
               int nseg, int tiles_per_seg, int ntiles, int idx_offset, int32_t *__restrict__ part_idx,
               int32_t *__restrict__ part_dist) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);   // SWIZZLE_128B atoms: 1024-B aligned
    uint8_t *smem_a = smem, *smem_b = smem + kTcSmemA;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + kTcSmemA + kTcStages * kTcSmemBStage);
    uint64_t *full = bars, *empty = bars + kTcStages, *a_full = bars + 2 * kTcStages, *a_empty = a_full + 1;
    uint64_t *tmem_full = a_empty + 1, *tmem_empty = tmem_full + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tmem_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int i = 0; i < kTcStages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        mbar_init(a_full, 1);
        mbar_init(a_empty, 1);
        for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 8); }
        mbar_init_fence();
    }
    if (warp == 1) {   // all 512 TMEM columns: two accumulator stages of 2 x 128
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0, it = 0;
            for (int item = blockIdx.x; item < nitems; item += gridDim.x, ++it) {
                const int mb = item / nseg, seg = item - mb * nseg;
                const int t0 = seg * tiles_per_seg, t1 = min(t0 + tiles_per_seg, ntiles);
                mbar_wait(a_empty, (it & 1) ^ 1);                   // the previous item's MMAs have read its query rows
                mbar_expect_tx(a_full, kTcSmemA);
                for (int h = 0; h < 2; ++h)
                    for (int kb = 0; kb < 2; ++kb)
                        tma_load_2d(smem_a + (h * 2 + kb) * kTcBoxBytes, &map_q, kb * 128, mb * kTcRowsPerItem + h * 128, a_full);
                for (int t = t0; t < t1; ++t) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    mbar_expect_tx(&full[stage], kTcSmemBStage);
                    uint8_t *dst = smem_b + stage * kTcSmemBStage;
                    tma_load_2d(dst, &map_t, 0, t * kTcTileN, &full[stage]);
                    tma_load_2d(dst + kTcBoxBytes, &map_t, 128, t * kTcTileN, &full[stage]);
                    if (++stage == kTcStages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0, it = 0, tcount = 0;
            for (int item = blockIdx.x; item < nitems; item += gridDim.x, ++it) {
                const int mb = item / nseg, seg = item - mb * nseg;
                const int t0 = seg * tiles_per_seg, t1 = min(t0 + tiles_per_seg, ntiles);
                mbar_wait(a_full, it & 1);
                for (int t = t0; t < t1; ++t, ++tcount) {
                    const uint32_t as = tcount & 1, aphase = (tcount >> 1) & 1;
                    mbar_wait(&tmem_empty[as], aphase ^ 1);          // the epilogue has drained this accumulator stage
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint8_t *bt = smem_b + stage * kTcSmemBStage;
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const uint32_t d = tmem_base + as * 256 + h * 128;
#pragma unroll
                        for (int kb = 0; kb < 2; ++kb) {
                            const uint64_t da = tc_smem_desc(smem_a + (h * 2 + kb) * kTcBoxBytes);
                            const uint64_t db = tc_smem_desc(bt + kb * kTcBoxBytes);
#pragma unroll
                            for (int k = 0; k < 4; ++k) tc_mma_i8(d, da + 2 * k, db + 2 * k, kTcIdesc, (kb | k) ? 1u : 0u);
                        }
                    }
                    tc_commit(&empty[stage]);                        // the train tile's smem slot is free once these MMAs retire
                    tc_commit(&tmem_full[as]);                       // ... and the accumulators are complete
                    if (++stage == kTcStages) { stage = 0; phase ^= 1; }
                }
                tc_commit(a_empty);
            }
        }
    } else {
        // ===== epilogue: thread = one query row =====
        const int h = (warp - 2) >> 2, q = warp & 3;                 // tcgen05.ld: warp w may touch TMEM lanes 32 (w % 4) ..
        const int row_in_item = h * 128 + q * 32 + lane;
        uint32_t tcount = 0;
        for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
            const int mb = item / nseg, seg = item - mb * nseg;
            const int t0 = seg * tiles_per_seg, t1 = min(t0 + tiles_per_seg, ntiles);
            int best = INT_MIN, best_i = -1, sec = INT_MIN, sec_i = -1;   // dot products: larger = closer
            for (int t = t0; t < t1; ++t, ++tcount) {
                const uint32_t as = tcount & 1, aphase = (tcount >> 1) & 1;
                mbar_wait(&tmem_full[as], aphase);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + as * 256 + h * 128;
#pragma unroll 1
                for (int c = 0; c < kTcTileN / 32; ++c) {
                    int v[32];
                    tc_ld32(taddr + c * 32, v);
                    tc_wait_ld();
                    int m = max3i(v[0], v[1], v[2]);
#pragma unroll
                    for (int j = 3; j + 1 < 32; j += 2) m = max3i(m, v[j], v[j + 1]);
                    m = max(m, v[31]);
                    if (m > sec) {                                    // rare: about 2 / (pairs seen so far)
                        const int n0 = t * kTcTileN + c * 32;
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const int d = v[j], n = n0 + j;
                            if (d > sec && n < nt) {                  // strict: a tie keeps the earlier (lower) index
                                if (d > best) { sec = best; sec_i = best_i; best = d; best_i = n; }
                                else { sec = d; sec_i = n; }
                            }
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tmem_empty[as]);
            }
            const int row = mb * kTcRowsPerItem + row_in_item;
            if (row < nq) {
                const int64_t o = ((int64_t)seg * nq + row) * 2;
                part_idx[o] = best_i >= 0 ? best_i + idx_offset : -1;
                part_dist[o] = best_i >= 0 ? (256 - best) >> 1 : INT_MAX;
                part_idx[o + 1] = sec_i >= 0 ? sec_i + idx_offset : -1;
                part_dist[o + 1] = sec_i >= 0 ? (256 - sec) >> 1 : INT_MAX;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
}

// ---- host side ----
EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
        else
            cudaGetLastError();
    }
    return fn;
}

// rows x 256 signed bytes, row-major; boxes of 128 rows x 128 bytes, SWIZZLE_128B, rows past the end read as zero
static bool make_row_map(CUtensorMap *map, const int8_t *base, int nrows) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return false;
    const cuuint64_t dims[2] = {256, (cuuint64_t)nrows};
    const cuuint64_t strides[1] = {256};
    const cuuint32_t box[2] = {128, 128};
    const cuuint32_t estr[2] = {1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, (void *)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

bool knn2_tc_supported(int nq, int nt) {
    const char *e = getenv("VSG_KNN_TC");   // 0 = never, 1 = auto (default), 2 = whenever the shapes allow (tests)
    const int mode = e ? atoi(e) : 1;
    if (mode == 0 || nt < 2 || nq < 1 || nt > (1 << 30)) return false;
    if (mode == 1 && ((int64_t)nq * nt < (1ll << 28) || nq < 256 || nt < 4096)) return false;   // small problems: the POPC kernel
    return encode_tiled_fn() != nullptr;
}

// kNN-2 of nq x nt descriptors on the tensor cores; out as vsg_knn2_dev.  Device buffers of the matcher: 14 expanded queries,
// 15 expanded train rows, 16 per-segment partial lists (slot 13 belongs to vsg_knn2_sharded, which calls this).
vsg_status knn2_tc_device(vsg_matcher *m, const uint8_t *q_dev, int nq, const uint8_t *t_dev, int nt, int offset, int *idx_dev,
                          int *dist_dev) {
    const int ntiles = (nt + kTcTileN - 1) / kTcTileN, n_mb = (nq + kTcRowsPerItem - 1) / kTcRowsPerItem;
    // segments: enough work items to balance the persistent CTAs (>= 8 items per CTA unless the tiles run out)
    int nseg = (8 * m->sm_count + n_mb - 1) / n_mb;
    nseg = std::max(1, std::min(nseg, std::min(ntiles, 64)));
    const int tiles_per_seg = (ntiles + nseg - 1) / nseg;
    nseg = (ntiles + tiles_per_seg - 1) / tiles_per_seg;
    const int nitems = n_mb * nseg;
    vsg_status st;
    if ((st = matcher_ensure(m, kSlotTcQuery, (size_t)nq * 256)) || (st = matcher_ensure(m, kSlotTcTrain, (size_t)nt * 256)) ||
        (st = matcher_ensure(m, kSlotTcParts, (size_t)nseg * nq * 2 * sizeof(int32_t) * 2)))
        return st;
    int8_t *q8 = (int8_t *)m->buf[kSlotTcQuery], *t8 = (int8_t *)m->buf[kSlotTcTrain];
    int32_t *part_idx = (int32_t *)m->buf[kSlotTcParts], *part_dist = part_idx + (size_t)nseg * nq * 2;
    cudaStream_t s = m->stream;
    expand_pm1_kernel<<<(unsigned)(((int64_t)nq * 8 + 255) / 256), 256, 0, s>>>((const uint32_t *)q_dev, nq, q8);
    expand_pm1_kernel<<<(unsigned)(((int64_t)nt * 8 + 255) / 256), 256, 0, s>>>((const uint32_t *)t_dev, nt, t8);
    CUtensorMap map_q, map_t;
    if (!make_row_map(&map_q, q8, nq) || !make_row_map(&map_t, t8, nt)) {
        set_error("knn2_tc: cuTensorMapEncodeTiled failed");
        return VSG_ERR_CUDA;
    }
    CK(cudaFuncSetAttribute(knn2_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmemBytes));
    const int grid = std::min(nitems, m->sm_count);
    knn2_tc_kernel<<<grid, kTcThreads, kTcSmemBytes, s>>>(map_q, map_t, nq, nt, nitems, nseg, tiles_per_seg, ntiles, offset, part_idx,
                                                         part_dist);
    count_launch(3);
    CK(cudaGetLastError());
    return launch_knn2_merge_parts(m, part_idx, part_dist, nseg, nq, idx_dev, dist_dev);
}

}  // namespace vsg
