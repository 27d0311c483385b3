// mappoint.cu — MapPoint::ComputeDistinctiveDescriptors for many map points at once, and the Lowe-ratio filter of
// Frame::ComputeStereoFishEyeMatches on top of the brute-force kNN-2.
//
// Reference (snt-arg/visual_sgraphs):
//   MapPoint::ComputeDistinctiveDescriptors    orb_slam3/src/MapPoint.cc:340-417
//     all observed descriptors of the point -> N x N Hamming distances (:383-394) -> per row the median
//     vDists[0.5 * (N - 1)] of the sorted row (:401-403) -> the row with the smallest median, first one on ties (:405-409)
//   Frame::ComputeStereoFishEyeMatches         orb_slam3/src/Frame.cc:1200-1208 (knnMatch k = 2, then
//     matches[0].distance < matches[1].distance * 0.7)
//
// A call splits its points at 32 observed descriptors:
// distinctive_warp_kernel: one warp per point with at most 32 descriptors (most of a keyframe's points have 2-30).  Lane i
//   holds row i in registers; the rows are broadcast by __shfl_sync and every distance is computed once into the warp's
//   32 x 32 16-bit tile in shared memory.  Lane i then reads its row back into registers and finds the k-th smallest entry
//   by a 9-step bisection on the value (distances are integers in [0, 256]); the warp minimum of (median << 16 | row)
//   keeps the first row on ties.
// distinctive_kernel: one CTA per point with more than 32 descriptors, over a compacted list of those points.  The point's
//   descriptors are staged in shared memory (up to 1024 rows); thread i owns row i of the distance matrix and runs the
//   same bisection, each step one pass of XOR + POPC over the row.  The CTA's best (median, row) pair is reduced with a
//   shared-memory atomicMin on (median << 16 | row).
#include <algorithm>
#include <cstring>
#include <vector>

#include "vsg_internal.cuh"

namespace vsg {

constexpr int kDistinctThreads = 128;
constexpr int kDistinctSmemRows = 1024;   // descriptors staged in shared memory (32 KB); longer lists are read from L2

__device__ __forceinline__ int hamming8(const uint32_t a[8], const uint4 b0, const uint4 b1) {
    return __popc(a[0] ^ b0.x) + __popc(a[1] ^ b0.y) + __popc(a[2] ^ b0.z) + __popc(a[3] ^ b0.w) +
           __popc(a[4] ^ b1.x) + __popc(a[5] ^ b1.y) + __popc(a[6] ^ b1.z) + __popc(a[7] ^ b1.w);
}

constexpr int kWarpRows = 32;                 // points with at most this many descriptors take the warp kernel
constexpr int kWarpsPerBlock = 8;
constexpr size_t kCopyPart = (size_t)1 << 20;

__global__ void __launch_bounds__(kWarpsPerBlock * 32) distinctive_warp_kernel(const uint4 *__restrict__ desc,
                                                                                const int *__restrict__ ptr, int npoints,
                                                                                int *__restrict__ best_out) {
    __shared__ uint16_t s_tile[kWarpsPerBlock][kWarpRows][kWarpRows];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int p = blockIdx.x * kWarpsPerBlock + warp;
    if (p >= npoints) return;
    const int begin = ptr[p], n = ptr[p + 1] - begin;
    if (n > kWarpRows) return;                                // distinctive_kernel's point
    if (n == 0) {
        if (lane == 0) best_out[p] = -1;                      // the reference returns without touching mDescriptor (:379)
        return;
    }
    uint32_t a[8] = {};
    if (lane < n) {
        const uint4 a0 = __ldg(desc + 2 * (size_t)(begin + lane)), a1 = __ldg(desc + 2 * (size_t)(begin + lane) + 1);
        a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w; a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
    }
    uint16_t (*tile)[kWarpRows] = s_tile[warp];
    for (int j = 0; j < n; ++j) {                             // tile[j][i] = dist(i, j): conflict-free stores and loads
        int d = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) d += __popc(a[w] ^ __shfl_sync(0xFFFFFFFFu, a[w], j));
        tile[j][lane] = (uint16_t)d;
    }
    __syncwarp();
    int row[kWarpRows];
#pragma unroll
    for (int j = 0; j < kWarpRows; ++j) row[j] = j < n ? tile[j][lane] : 0x7FFF;   // padding never counts as <= mid
    const int k = (int)(0.5 * (n - 1));                      // vDists[0.5 * (N - 1)] (:403)
    int lo = 0, hi = 256;                                     // smallest v with #{j : dist(i, j) <= v} >= k + 1
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        int cnt = 0;
#pragma unroll
        for (int j = 0; j < kWarpRows; ++j) cnt += row[j] <= mid;
        if (cnt >= k + 1) hi = mid; else lo = mid + 1;
    }
    const unsigned best = __reduce_min_sync(0xFFFFFFFFu, lane < n ? ((unsigned)lo << 16) | (unsigned)lane : 0xFFFFFFFFu);
    if (lane == 0) best_out[p] = (int)(best & 0xFFFFu);
}

__global__ void __launch_bounds__(kDistinctThreads) distinctive_kernel(const uint4 *__restrict__ desc,
                                                                       const int *__restrict__ ptr,
                                                                       const int *__restrict__ points,
                                                                       int *__restrict__ best_out) {
    extern __shared__ uint4 s_desc[];
    __shared__ unsigned s_best;
    const int p = points[blockIdx.x];
    const int begin = ptr[p], n = ptr[p + 1] - begin;       // n > kWarpRows
    const uint4 *d = desc + 2 * (size_t)begin;
    const bool staged = n <= kDistinctSmemRows;
    if (staged)
        for (int i = threadIdx.x; i < 2 * n; i += kDistinctThreads) s_desc[i] = __ldg(d + i);
    if (threadIdx.x == 0) s_best = 0xFFFFFFFFu;
    __syncthreads();
    const uint4 *rows = staged ? s_desc : d;
    const int k = (int)(0.5 * (n - 1));                      // vDists[0.5 * (N - 1)] (:403)
    for (int i = threadIdx.x; i < n; i += kDistinctThreads) {
        uint32_t a[8];
        {
            const uint4 a0 = rows[2 * i], a1 = rows[2 * i + 1];
            a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w; a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
        }
        // smallest v with #{j : dist(i, j) <= v} >= k + 1  ==  the k-th entry of the sorted row
        int lo = 0, hi = 256;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            int cnt = 0;
            for (int j = 0; j < n; ++j) cnt += hamming8(a, rows[2 * j], rows[2 * j + 1]) <= mid;
            if (cnt >= k + 1) hi = mid; else lo = mid + 1;
        }
        atomicMin(&s_best, ((unsigned)lo << 16) | (unsigned)min(i, 0xFFFF));
    }
    __syncthreads();
    if (threadIdx.x == 0) best_out[p] = (int)(s_best & 0xFFFFu);
}

}  // namespace vsg

using namespace vsg;

extern "C" {

vsg_status vsg_distinctive_descriptors(vsg_matcher *m, const uint8_t *descriptors, const int32_t *ptr, int npoints,
                                       int32_t *best_out) {
    if (!m || npoints < 0 || (npoints > 0 && (!ptr || !best_out))) return VSG_ERR_INVALID;
    if (npoints == 0) return VSG_OK;
    const int total = ptr[npoints];
    int longest = 0;
    for (int p = 0; p < npoints; ++p) {
        if (ptr[p + 1] < ptr[p]) { set_error("vsg_distinctive_descriptors: ptr must be non-decreasing"); return VSG_ERR_INVALID; }
        longest = std::max(longest, ptr[p + 1] - ptr[p]);
    }
    if (longest > 65535) { set_error("vsg_distinctive_descriptors: more than 65535 observations of one point"); return VSG_ERR_INVALID; }
    if (total > 0 && !descriptors) return VSG_ERR_INVALID;
    std::vector<int> longp;                                  // the points of distinctive_kernel
    for (int p = 0; p < npoints; ++p)
        if (ptr[p + 1] - ptr[p] > kWarpRows) longp.push_back(p);
    const int nlong = (int)longp.size();
    // one pinned staging block: descriptors | ptr | long points, then the results on their way back
    const size_t o_ptr = (size_t)total * 32, o_long = o_ptr + (size_t)(npoints + 1) * 4, in_bytes = o_long + (size_t)nlong * 4,
                 o_out = (in_bytes + 15) & ~(size_t)15;
    CK(cudaSetDevice(m->device));
    vsg_status st;
    if ((st = matcher_ensure(m, kSlotArg1, in_bytes)) || (st = matcher_ensure(m, kSlotOut, (size_t)npoints * 4)) ||
        (st = matcher_ensure_host(m, kHostDistinctive, o_out + (size_t)npoints * 4)))
        return st;
    uint8_t *h = (uint8_t *)m->hbuf[kHostDistinctive], *d = (uint8_t *)m->buf[kSlotArg1];
    memcpy(h + o_ptr, ptr, (size_t)(npoints + 1) * 4);
    if (nlong) memcpy(h + o_long, longp.data(), (size_t)nlong * 4);
    cudaStream_t s = m->stream;
    int *out = (int *)m->buf[kSlotOut];
    // one copy per MB: in a larger call the staging of a part overlaps the copy of the part before it
    for (size_t off = 0; off < in_bytes; off += kCopyPart) {
        const size_t end = std::min(in_bytes, off + kCopyPart);
        if (off < o_ptr) memcpy(h + off, descriptors + off, std::min(end, o_ptr) - off);
        CK(cudaMemcpyAsync(d + off, h + off, end - off, cudaMemcpyHostToDevice, s));
    }
    if (nlong < npoints) {
        distinctive_warp_kernel<<<(npoints + kWarpsPerBlock - 1) / kWarpsPerBlock, kWarpsPerBlock * 32, 0, s>>>(
            (const uint4 *)d, (const int *)(d + o_ptr), npoints, out);
        count_launch();
        CK(cudaGetLastError());
    }
    if (nlong) {
        const size_t smem = (size_t)std::min(longest, kDistinctSmemRows) * 32;
        if (smem > 48 * 1024) CK(cudaFuncSetAttribute(distinctive_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        distinctive_kernel<<<nlong, kDistinctThreads, smem, s>>>((const uint4 *)d, (const int *)(d + o_ptr),
                                                                 (const int *)(d + o_long), out);
        count_launch();
        CK(cudaGetLastError());
    }
    CK(cudaMemcpyAsync(h + o_out, out, (size_t)npoints * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    memcpy(best_out, h + o_out, (size_t)npoints * 4);
    return VSG_OK;
}

vsg_status vsg_knn2_ratio(vsg_matcher *m, const uint8_t *query, int nq, const uint8_t *train, int nt, float ratio,
                          int32_t *match_out, int32_t *dist_out) {
    if (!m || nq < 0 || nt < 0 || (nq > 0 && !match_out)) return VSG_ERR_INVALID;
    std::vector<int32_t> idx((size_t)std::max(nq, 1) * 2), dist((size_t)std::max(nq, 1) * 2);
    vsg_status st = vsg_knn2(m, query, nq, train, nt, 0, idx.data(), dist.data());
    if (st != VSG_OK) return st;
    for (int i = 0; i < nq; ++i) {
        // (*it).size() >= 2 && (*it)[0].distance < (*it)[1].distance * 0.7   (DMatch::distance is a float; the
        // reference's literal 0.7 is a double, so the product and the comparison are done in double)
        const bool two = idx[2 * i + 1] >= 0;
        const bool good = two && (double)(float)dist[2 * i] < (double)(float)dist[2 * i + 1] * (double)ratio;
        match_out[i] = good ? idx[2 * i] : -1;
        if (dist_out) dist_out[i] = idx[2 * i] >= 0 ? dist[2 * i] : -1;
    }
    return VSG_OK;
}

}  // extern "C"
