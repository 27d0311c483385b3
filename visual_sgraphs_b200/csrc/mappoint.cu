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
// distinctive_kernel: one CTA per map point.  The point's descriptors are staged in shared memory; thread i owns row
// i of the distance matrix and finds its median without storing or sorting the row: distances are integers in
// [0, 256], so the k-th smallest is found by a 9-step bisection on the value, each step one pass of XOR + POPC over
// the row.  The CTA's best (median, row) pair is reduced with a shared-memory atomicMin on (median << 16 | row).
#include <algorithm>
#include <vector>

#include "vsg_internal.cuh"

namespace vsg {

constexpr int kDistinctThreads = 128;
constexpr int kDistinctSmemRows = 1024;   // descriptors staged in shared memory (32 KB); longer lists are read from L2

__device__ __forceinline__ int hamming8(const uint32_t a[8], const uint4 b0, const uint4 b1) {
    return __popc(a[0] ^ b0.x) + __popc(a[1] ^ b0.y) + __popc(a[2] ^ b0.z) + __popc(a[3] ^ b0.w) +
           __popc(a[4] ^ b1.x) + __popc(a[5] ^ b1.y) + __popc(a[6] ^ b1.z) + __popc(a[7] ^ b1.w);
}

__global__ void __launch_bounds__(kDistinctThreads) distinctive_kernel(const uint4 *__restrict__ desc,
                                                                       const int *__restrict__ ptr, int npoints,
                                                                       int *__restrict__ best_out) {
    extern __shared__ uint4 s_desc[];
    __shared__ unsigned s_best;
    const int p = blockIdx.x;
    const int begin = ptr[p], n = ptr[p + 1] - begin;
    if (n <= 0) {
        if (threadIdx.x == 0) best_out[p] = -1;              // the reference returns without touching mDescriptor (:354,379)
        return;
    }
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
    CK(cudaSetDevice(m->device));
    vsg_status st;
    if ((st = matcher_ensure(m, kSlotArg1, (size_t)std::max(total, 1) * 32)) || (st = matcher_ensure(m, kSlotArg3, (size_t)(npoints + 1) * 4)) ||
        (st = matcher_ensure(m, kSlotOut, (size_t)npoints * 4)))
        return st;
    cudaStream_t s = m->stream;
    if (total > 0) CK(cudaMemcpyAsync(m->buf[kSlotArg1], descriptors, (size_t)total * 32, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(m->buf[kSlotArg3], ptr, (size_t)(npoints + 1) * 4, cudaMemcpyHostToDevice, s));
    const size_t smem = (size_t)std::min(longest, kDistinctSmemRows) * 32;
    if (smem > 48 * 1024) CK(cudaFuncSetAttribute(distinctive_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    distinctive_kernel<<<npoints, kDistinctThreads, smem, s>>>((const uint4 *)m->buf[kSlotArg1], (const int *)m->buf[kSlotArg3], npoints,
                                                             (int *)m->buf[kSlotOut]);
    count_launch();
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(best_out, m->buf[kSlotOut], (size_t)npoints * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
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
