// stereo.cu — Frame::ComputeStereoMatches on the device pyramids of the two extractors.
//
// Reference (snt-arg/visual_sgraphs): orb_slam3/src/Frame.cc:957-1127.
//   :969-984   right keypoints are listed in every integer row of [floor(y - r), ceil(y + r)], r = 2*scale[octave]
//   :996-1040  per left keypoint: candidates of row (size_t)vL, octave within +-1, uR in [uL - maxD, uL],
//              best Hamming distance starting from TH_HIGH with strict '<' (first candidate wins ties)
//   :1043-1079 if best < (TH_HIGH+TH_LOW)/2: 11x11 L1 norm (cv::norm NORM_L1) against the right level at 11
//              horizontal offsets; :1081-1092 parabola fit; :1095-1109 disparity gate
//   :1113-1126 sort (SAD, iL), reject SAD >= 1.5*1.4*median
//
// stereo_search_kernel: one thread per left keypoint.  Instead of materialising the row table it tests every
//   right keypoint's band against the left keypoint's row, in right-index order — the same candidates in the
//   same order as vRowIndices[(size_t)vL].  Right keypoints are staged in shared memory.
// stereo_sad_kernel: one warp per left keypoint; lanes stride over the 121 patch pixels, 11 offsets each.
// The final median rejection is a sort of <= N pairs and runs on the host inside the entry point.
#include <algorithm>
#include <climits>
#include <cmath>
#include <vector>

#include "vsg_internal.cuh"

namespace vsg {

struct RightKp {          // what the row-band test needs of a right keypoint
    float x;
    int minr, maxr;       // floor(y - r), ceil(y + r)
    int octave;
};

struct LevelPlane {
    const uint8_t *base;  // frame-adjusted
    int pitch, w, h;
};
struct StereoPlanes {
    LevelPlane l[kMaxLevels], r[kMaxLevels];
    float scale[kMaxLevels], inv_scale[kMaxLevels];
};

__device__ __forceinline__ int hamming256(const uint4 &a0, const uint4 &a1, const uint4 &b0, const uint4 &b1) {
    return __popc(a0.x ^ b0.x) + __popc(a0.y ^ b0.y) + __popc(a0.z ^ b0.z) + __popc(a0.w ^ b0.w) +
           __popc(a1.x ^ b1.x) + __popc(a1.y ^ b1.y) + __popc(a1.z ^ b1.z) + __popc(a1.w ^ b1.w);
}

__global__ void stereo_search_kernel(const vsg_keypoint *__restrict__ keys_l, const uint4 *__restrict__ desc_l, int n_l,
                                     const RightKp *__restrict__ right, const uint4 *__restrict__ desc_r, int n_r,
                                     int n_rows, float max_d, int *__restrict__ best_dist, int *__restrict__ best_idx) {
    extern __shared__ RightKp s_right[];
    for (int i = threadIdx.x; i < n_r; i += blockDim.x) s_right[i] = right[i];
    __syncthreads();
    const int il = blockIdx.x * blockDim.x + threadIdx.x;
    if (il >= n_l) return;
    const vsg_keypoint kpl = keys_l[il];
    int bd = 100, bi = 0;                                     // bestDist = TH_HIGH (:1013)
    const float vl = kpl.y, ul = kpl.x;
    const int row = (int)vl;                                  // vRowIndices[vL] (:1002)
    const float min_u = ul - max_d, max_u = ul;               // minD = 0 (:988,1007-1008)
    if (row >= 0 && row < n_rows && !(max_u < 0)) {
        const uint4 la = __ldg(desc_l + 2 * il), lb = __ldg(desc_l + 2 * il + 1);
        for (int ir = 0; ir < n_r; ++ir) {
            const RightKp k = s_right[ir];
            if (row < k.minr || row > k.maxr) continue;       // not listed in this row
            if (k.octave < kpl.octave - 1 || k.octave > kpl.octave + 1) continue;
            if (k.x >= min_u && k.x <= max_u) {
                const int d = hamming256(la, lb, __ldg(desc_r + 2 * ir), __ldg(desc_r + 2 * ir + 1));
                if (d < bd) { bd = d; bi = ir; }
            }
        }
    }
    best_dist[il] = bd;
    best_idx[il] = bi;
}

// out[il] = {SAD of the best offset (or -1 if rejected), bestuR bits, disparity-ok flag}
__global__ void stereo_sad_kernel(StereoPlanes P, const vsg_keypoint *__restrict__ keys_l, int n_l,
                                  const RightKp *__restrict__ right, const int *__restrict__ best_dist,
                                  const int *__restrict__ best_idx, float max_d, float mbf, int *__restrict__ sad_out,
                                  float *__restrict__ u_right, float *__restrict__ depth) {
    const int il = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (il >= n_l) return;
    if (lane == 0) { sad_out[il] = -1; u_right[il] = -1.0f; depth[il] = -1.0f; }
    if (best_dist[il] >= 75) return;                          // thOrbDist = (TH_HIGH + TH_LOW) / 2 (:962,1043)
    const vsg_keypoint kpl = keys_l[il];
    const int oct = kpl.octave;
    const float ur0 = right[best_idx[il]].x;
    const float sf = P.inv_scale[oct];
    const float sul = roundf(__fmul_rn(kpl.x, sf)), svl = roundf(__fmul_rn(kpl.y, sf)), sur0 = roundf(__fmul_rn(ur0, sf));
    const int w = 5, L = 5;
    const LevelPlane pl = P.l[oct], pr = P.r[oct];
    const float iniu = sur0 + L - w, endu = sur0 + L + w + 1;
    if (iniu < 0 || endu >= pr.w) return;                     // :1062-1065
    const int y0 = (int)(svl - w), xl0 = (int)(sul - w), xr0 = (int)(sur0 - L - w);
    // The 11 x 11 left patch and the 11 x 21 right strip must lie inside the level: the reference's rowRange / colRange throw
    // a cv::Exception for a keypoint this close to the border (:1054, :1069); extractor keypoints never are (>= 19 px from
    // every edge), caller-supplied ones get "no match" instead of an out-of-bounds read.
    if (y0 < 0 || y0 + 2 * w >= pl.h || y0 + 2 * w >= pr.h || xl0 < 0 || xl0 + 2 * w >= pl.w || xr0 < 0) return;
    int sad[11];
#pragma unroll
    for (int k = 0; k < 11; ++k) sad[k] = 0;
    for (int p = lane; p < 121; p += 32) {
        const int dy = p / 11, dx = p - dy * 11;
        const int a = __ldg(pl.base + (int64_t)(y0 + dy) * pl.pitch + xl0 + dx);
        const uint8_t *rrow = pr.base + (int64_t)(y0 + dy) * pr.pitch + xr0 + dx;
#pragma unroll
        for (int k = 0; k < 11; ++k) sad[k] += abs(a - (int)__ldg(rrow + k));
    }
#pragma unroll
    for (int k = 0; k < 11; ++k)
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) sad[k] += __shfl_xor_sync(0xffffffffu, sad[k], d);
    if (lane != 0) return;
    int best = INT_MAX, best_inc = 0;                         // float dist < int bestDist: exact for these magnitudes
#pragma unroll
    for (int k = 0; k < 11; ++k)
        if (sad[k] < best) { best = sad[k]; best_inc = k - L; }
    if (best_inc == -L || best_inc == L) return;              // :1081
    float d1 = 0.f, d2 = 0.f, d3 = 0.f;
#pragma unroll
    for (int k = 1; k < 10; ++k)
        if (k - L == best_inc) { d1 = (float)sad[k - 1]; d2 = (float)sad[k]; d3 = (float)sad[k + 1]; }
    const float delta = __fdiv_rn(__fsub_rn(d1, d3), __fmul_rn(2.0f, __fsub_rn(__fadd_rn(d1, d3), __fmul_rn(2.0f, d2))));
    if (delta < -1 || delta > 1) return;                      // :1089
    float best_ur = __fmul_rn(P.scale[oct], __fadd_rn(__fadd_rn(sur0, (float)best_inc), delta));   // :1095
    float disparity = __fsub_rn(kpl.x, best_ur);
    if (disparity >= 0.f && disparity < max_d) {              // :1097-1109
        if (disparity <= 0) {
            disparity = 0.01f;                                // (float)0.01
            best_ur = (float)((double)kpl.x - 0.01);
        }
        depth[il] = __fdiv_rn(mbf, disparity);
        u_right[il] = best_ur;
        sad_out[il] = best;
    }
}

// ---- batched variant: pairs (2p, 2p+1) of one extractor batch, everything device-resident ----
struct BatchPlanes {          // frame-0 base of every level + strides; frame f of level l = base[l] + f * stride[l]
    const uint8_t *base[kMaxLevels];
    int64_t stride[kMaxLevels];
    int pitch[kMaxLevels], w[kMaxLevels], h[kMaxLevels];
    float scale[kMaxLevels], inv_scale[kMaxLevels];
    int n_rows;
};

__global__ void stereo_search_batch_kernel(BatchPlanes P, const vsg_keypoint *__restrict__ kps, const uint4 *__restrict__ desc,
                                           const int *__restrict__ n_kp, int out_cap, float max_d,
                                           int *__restrict__ best_dist, int *__restrict__ best_idx) {
    extern __shared__ RightKp s_right[];
    const int pair = blockIdx.y;
    const vsg_keypoint *keys_l = kps + (size_t)(2 * pair) * out_cap, *keys_r = keys_l + out_cap;
    const uint4 *desc_l = desc + (size_t)(2 * pair) * out_cap * 2, *desc_r = desc_l + (size_t)out_cap * 2;
    const int n_l = min(n_kp[2 * pair], out_cap), n_r = min(n_kp[2 * pair + 1], out_cap);
    for (int i = threadIdx.x; i < n_r; i += blockDim.x) {                       // :973-984
        const vsg_keypoint k = keys_r[i];
        const float r = __fmul_rn(2.0f, P.scale[k.octave]);
        RightKp rk;
        rk.x = k.x;
        rk.maxr = (int)ceilf(__fadd_rn(k.y, r));
        rk.minr = (int)floorf(__fsub_rn(k.y, r));
        rk.octave = k.octave;
        s_right[i] = rk;
    }
    __syncthreads();
    const int il = blockIdx.x * blockDim.x + threadIdx.x;
    if (il >= n_l) return;
    const vsg_keypoint kpl = keys_l[il];
    int bd = 100, bi = 0;
    const int row = (int)kpl.y;
    const float min_u = kpl.x - max_d, max_u = kpl.x;
    if (row >= 0 && row < P.n_rows && !(max_u < 0)) {
        const uint4 la = __ldg(desc_l + 2 * il), lb = __ldg(desc_l + 2 * il + 1);
        for (int ir = 0; ir < n_r; ++ir) {
            const RightKp k = s_right[ir];
            if (row < k.minr || row > k.maxr) continue;
            if (k.octave < kpl.octave - 1 || k.octave > kpl.octave + 1) continue;
            if (k.x >= min_u && k.x <= max_u) {
                const int d = hamming256(la, lb, __ldg(desc_r + 2 * ir), __ldg(desc_r + 2 * ir + 1));
                if (d < bd) { bd = d; bi = ir; }
            }
        }
    }
    best_dist[(size_t)pair * out_cap + il] = bd;
    best_idx[(size_t)pair * out_cap + il] = bi;
}

__global__ void stereo_sad_batch_kernel(BatchPlanes P, const vsg_keypoint *__restrict__ kps, const int *__restrict__ n_kp,
                                        int out_cap, const int *__restrict__ best_dist, const int *__restrict__ best_idx,
                                        float max_d, float mbf, int *__restrict__ sad_out, float *__restrict__ u_right,
                                        float *__restrict__ depth) {
    const int pair = blockIdx.y;
    const int il = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (il >= out_cap) return;
    const size_t o = (size_t)pair * out_cap + il;
    if (lane == 0) { sad_out[o] = -1; u_right[o] = -1.0f; depth[o] = -1.0f; }
    if (il >= min(n_kp[2 * pair], out_cap)) return;
    if (best_dist[o] >= 75) return;
    const vsg_keypoint *keys_l = kps + (size_t)(2 * pair) * out_cap, *keys_r = keys_l + out_cap;
    const vsg_keypoint kpl = keys_l[il];
    const int oct = kpl.octave;
    const float ur0 = keys_r[best_idx[o]].x;
    const float sf = P.inv_scale[oct];
    const float sul = roundf(__fmul_rn(kpl.x, sf)), svl = roundf(__fmul_rn(kpl.y, sf)), sur0 = roundf(__fmul_rn(ur0, sf));
    const int w = 5, L = 5;
    const float iniu = sur0 + L - w, endu = sur0 + L + w + 1;
    if (iniu < 0 || endu >= P.w[oct]) return;
    const uint8_t *pl = P.base[oct] + (int64_t)(2 * pair) * P.stride[oct], *pr = pl + P.stride[oct];
    const int pitch = P.pitch[oct];
    const int y0 = (int)(svl - w), xl0 = (int)(sul - w), xr0 = (int)(sur0 - L - w);
    if (y0 < 0 || y0 + 2 * w >= P.h[oct] || xl0 < 0 || xl0 + 2 * w >= P.w[oct] || xr0 < 0) return;   // see stereo_sad_kernel
    int sad[11];
#pragma unroll
    for (int k = 0; k < 11; ++k) sad[k] = 0;
    for (int p = lane; p < 121; p += 32) {
        const int dy = p / 11, dx = p - dy * 11;
        const int a = __ldg(pl + (int64_t)(y0 + dy) * pitch + xl0 + dx);
        const uint8_t *rrow = pr + (int64_t)(y0 + dy) * pitch + xr0 + dx;
#pragma unroll
        for (int k = 0; k < 11; ++k) sad[k] += abs(a - (int)__ldg(rrow + k));
    }
#pragma unroll
    for (int k = 0; k < 11; ++k)
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) sad[k] += __shfl_xor_sync(0xffffffffu, sad[k], d);
    if (lane != 0) return;
    int best = INT_MAX, best_inc = 0;
#pragma unroll
    for (int k = 0; k < 11; ++k)
        if (sad[k] < best) { best = sad[k]; best_inc = k - L; }
    if (best_inc == -L || best_inc == L) return;
    float d1 = 0.f, d2 = 0.f, d3 = 0.f;
#pragma unroll
    for (int k = 1; k < 10; ++k)
        if (k - L == best_inc) { d1 = (float)sad[k - 1]; d2 = (float)sad[k]; d3 = (float)sad[k + 1]; }
    const float delta = __fdiv_rn(__fsub_rn(d1, d3), __fmul_rn(2.0f, __fsub_rn(__fadd_rn(d1, d3), __fmul_rn(2.0f, d2))));
    if (delta < -1 || delta > 1) return;
    float best_ur = __fmul_rn(P.scale[oct], __fadd_rn(__fadd_rn(sur0, (float)best_inc), delta));
    float disparity = __fsub_rn(kpl.x, best_ur);
    if (disparity >= 0.f && disparity < max_d) {
        if (disparity <= 0) {
            disparity = 0.01f;
            best_ur = (float)((double)kpl.x - 0.01);
        }
        depth[o] = __fdiv_rn(mbf, disparity);
        u_right[o] = best_ur;
        sad_out[o] = best;
    }
}

// :1113-1126 per pair: median = the (count / 2)-th smallest SAD of the accepted matches (0-based, as in the sorted
// vDistIdx), found by bisection on the integer SAD value; every match with SAD >= 1.5f * 1.4f * median is dropped
// (the reference walks the sorted vector from the back until the first SAD below the threshold: the same set).
__global__ void __launch_bounds__(256) stereo_median_kernel(int out_cap, const int *__restrict__ sad, float *__restrict__ u_right,
                                                            float *__restrict__ depth) {
    __shared__ int s_cnt;
    const int pair = blockIdx.x, tid = threadIdx.x;
    const int *s = sad + (size_t)pair * out_cap;
    int valid = 0;
    for (int i = tid; i < out_cap; i += 256) valid += s[i] >= 0;
    if (tid == 0) s_cnt = 0;
    __syncthreads();
    atomicAdd(&s_cnt, valid);
    __syncthreads();
    const int total = s_cnt;
    if (total == 0) return;
    const int k = total / 2;
    int lo = 0, hi = 121 * 255;                                 // smallest v with #{sad <= v} >= k + 1
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        __syncthreads();
        if (tid == 0) s_cnt = 0;
        __syncthreads();
        int c = 0;
        for (int i = tid; i < out_cap; i += 256) c += (s[i] >= 0 && s[i] <= mid);
        atomicAdd(&s_cnt, c);
        __syncthreads();
        if (s_cnt >= k + 1) hi = mid; else lo = mid + 1;
    }
    const float th = __fmul_rn(__fmul_rn(1.5f, 1.4f), (float)lo);
    for (int i = tid; i < out_cap; i += 256)
        if (s[i] >= 0 && !((float)s[i] < th)) {
            u_right[(size_t)pair * out_cap + i] = -1.0f;
            depth[(size_t)pair * out_cap + i] = -1.0f;
        }
}

}  // namespace vsg

using namespace vsg;

extern "C" vsg_status vsg_stereo_match(vsg_matcher *m, vsg_extractor *left, vsg_extractor *right, int frame_l, int frame_r,
                                       const vsg_keypoint *keys_l, const uint8_t *desc_l, int n_l,
                                       const vsg_keypoint *keys_r, const uint8_t *desc_r, int n_r, float mb, float mbf,
                                       float *u_right_out, float *depth_out) {
    if (!m || !left || !right || n_l < 0 || n_r < 0 || !u_right_out || !depth_out ||
        (n_l > 0 && (!keys_l || !desc_l)) || (n_r > 0 && (!keys_r || !desc_r)))
        return VSG_ERR_INVALID;
    PyramidRef pl, pr;
    if (!extractor_pyramid(left, &pl) || !extractor_pyramid(right, &pr) || frame_l < 0 || frame_l >= pl.nframes ||
        frame_r < 0 || frame_r >= pr.nframes || pl.device != m->device || pr.device != m->device ||
        pl.geom->nlevels != pr.geom->nlevels) {
        set_error("vsg_stereo_match: both extractors must have run on the matcher's device with the same level count");
        return VSG_ERR_INVALID;
    }
    for (int i = 0; i < n_l; ++i) { u_right_out[i] = -1.0f; depth_out[i] = -1.0f; }
    if (n_l == 0 || n_r == 0) return VSG_OK;
    CK(cudaSetDevice(m->device));
    // the extractors' streams must have finished producing the pyramids
    CK(cudaStreamSynchronize(pl.stream));
    CK(cudaStreamSynchronize(pr.stream));
    const int nl = pl.geom->nlevels;
    StereoPlanes P;
    for (int l = 0; l < nl; ++l) {
        const LevelGeom &GL = pl.geom->lv[l], &GR = pr.geom->lv[l];
        if (l == 0) {
            P.l[l] = LevelPlane{pl.lvl0_base + (int64_t)frame_l * pl.lvl0_stride, pl.lvl0_pitch, GL.w, GL.h};
            P.r[l] = LevelPlane{pr.lvl0_base + (int64_t)frame_r * pr.lvl0_stride, pr.lvl0_pitch, GR.w, GR.h};
        } else {
            P.l[l] = LevelPlane{pl.pyr + GL.plane_offset + (int64_t)frame_l * GL.plane_stride, GL.pitch, GL.w, GL.h};
            P.r[l] = LevelPlane{pr.pyr + GR.plane_offset + (int64_t)frame_r * GR.plane_stride, GR.pitch, GR.w, GR.h};
        }
        P.scale[l] = pl.scale[l];
        P.inv_scale[l] = pl.inv_scale[l];
    }
    const int n_rows = pl.geom->lv[0].h;                      // mvImagePyramid[0].rows (:964)
    std::vector<RightKp> rk(n_r);
    for (int i = 0; i < n_r; ++i) {                           // :973-984
        const int oct = keys_r[i].octave;
        if (oct < 0 || oct >= nl) { set_error("vsg_stereo_match: right keypoint %d has octave %d", i, oct); return VSG_ERR_INVALID; }
        const float r = 2.0f * pl.scale[oct];
        rk[i].x = keys_r[i].x;
        rk[i].maxr = (int)std::ceil(keys_r[i].y + r);
        rk[i].minr = (int)std::floor(keys_r[i].y - r);
        rk[i].octave = oct;
    }
    for (int i = 0; i < n_l; ++i)
        if (keys_l[i].octave < 0 || keys_l[i].octave >= nl) { set_error("vsg_stereo_match: left keypoint %d has octave %d", i, keys_l[i].octave); return VSG_ERR_INVALID; }
    vsg_status st;
    // best dist/idx/sad: 3 x n_l ints; u_right/depth: 2 x n_l floats
    if ((st = matcher_ensure(m, kSlotArg1, (size_t)n_l * sizeof(vsg_keypoint))) || (st = matcher_ensure(m, kSlotArg2, (size_t)n_l * 32)) ||
        (st = matcher_ensure(m, kSlotArg3, (size_t)n_r * sizeof(RightKp))) || (st = matcher_ensure(m, kSlotArg4, (size_t)n_r * 32)) ||
        (st = matcher_ensure(m, kSlotOut, (size_t)n_l * 12)) || (st = matcher_ensure(m, kSlotAreaQueries, (size_t)n_l * 8)))
        return st;
    cudaStream_t s = m->stream;
    CK(cudaMemcpyAsync(m->buf[kSlotArg1], keys_l, (size_t)n_l * sizeof(vsg_keypoint), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(m->buf[kSlotArg2], desc_l, (size_t)n_l * 32, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(m->buf[kSlotArg3], rk.data(), (size_t)n_r * sizeof(RightKp), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(m->buf[kSlotArg4], desc_r, (size_t)n_r * 32, cudaMemcpyHostToDevice, s));
    int *bd = (int *)m->buf[kSlotOut], *bi = bd + n_l, *sad = bi + n_l;
    float *ur = (float *)m->buf[kSlotAreaQueries], *dp = ur + n_l;
    const float max_d = mbf / mb;                             // :987-989
    const size_t smem = (size_t)n_r * sizeof(RightKp);
    if (smem > 200 * 1024) { set_error("vsg_stereo_match: too many right keypoints (%d)", n_r); return VSG_ERR_INVALID; }
    if (smem > 48 * 1024) CK(cudaFuncSetAttribute(stereo_search_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    stereo_search_kernel<<<(n_l + 127) / 128, 128, smem, s>>>((const vsg_keypoint *)m->buf[kSlotArg1], (const uint4 *)m->buf[kSlotArg2], n_l,
                                                             (const RightKp *)m->buf[kSlotArg3], (const uint4 *)m->buf[kSlotArg4], n_r,
                                                             n_rows, max_d, bd, bi);
    stereo_sad_kernel<<<(n_l + 7) / 8, 256, 0, s>>>(P, (const vsg_keypoint *)m->buf[kSlotArg1], n_l, (const RightKp *)m->buf[kSlotArg3], bd, bi,
                                                   max_d, mbf, sad, ur, dp);
    count_launch(2);
    CK(cudaGetLastError());
    std::vector<int> sad_h(n_l);
    CK(cudaMemcpyAsync(sad_h.data(), sad, (size_t)n_l * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(u_right_out, ur, (size_t)n_l * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(depth_out, dp, (size_t)n_l * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    // :1113-1126 median-based rejection (the sort is over (SAD, iL) pairs: a total order)
    std::vector<std::pair<int, int>> dist_idx;
    for (int i = 0; i < n_l; ++i)
        if (sad_h[i] >= 0) dist_idx.push_back(std::make_pair(sad_h[i], i));
    if (dist_idx.empty()) return VSG_OK;                      // the reference reads vDistIdx[0] here (SURVEY C#12)
    std::sort(dist_idx.begin(), dist_idx.end());
    const float median = (float)dist_idx[dist_idx.size() / 2].first;
    const float th_dist = 1.5f * 1.4f * median;
    for (int i = (int)dist_idx.size() - 1; i >= 0; --i) {
        if (dist_idx[i].first < th_dist) break;
        u_right_out[dist_idx[i].second] = -1;
        depth_out[dist_idx[i].second] = -1;
    }
    return VSG_OK;
}

extern "C" vsg_status vsg_stereo_match_batch(vsg_matcher *m, vsg_extractor *ex, int npairs, float mb, float mbf,
                                             float *u_right_out, float *depth_out, int capacity) {
    if (!m || !ex || npairs < 0 || (npairs > 0 && (!u_right_out || !depth_out))) return VSG_ERR_INVALID;
    PyramidRef pr;
    if (!extractor_pyramid(ex, &pr) || !pr.kps_dev || pr.device != m->device || 2 * npairs > pr.nframes) {
        set_error("vsg_stereo_match_batch: the extractor's last call must be a host-pointer batch of >= 2 * npairs frames on the "
                  "matcher's device (frames 2p / 2p+1 = left / right image of pair p)");
        return VSG_ERR_INVALID;
    }
    if (capacity < pr.out_cap) {
        set_error("vsg_stereo_match_batch: capacity %d < vsg_extractor_max_keypoints() = %d", capacity, pr.out_cap);
        return VSG_ERR_CAPACITY;
    }
    if (npairs == 0) return VSG_OK;
    CK(cudaSetDevice(m->device));
    CK(cudaStreamSynchronize(pr.stream));
    const int nl = pr.geom->nlevels, cap = pr.out_cap;
    BatchPlanes P;
    for (int l = 0; l < nl; ++l) {
        const LevelGeom &G = pr.geom->lv[l];
        if (l == 0) { P.base[l] = pr.lvl0_base; P.stride[l] = pr.lvl0_stride; P.pitch[l] = pr.lvl0_pitch; }
        else { P.base[l] = pr.pyr + G.plane_offset; P.stride[l] = G.plane_stride; P.pitch[l] = G.pitch; }
        P.w[l] = G.w;
        P.h[l] = G.h;
        P.scale[l] = pr.scale[l];
        P.inv_scale[l] = pr.inv_scale[l];
    }
    P.n_rows = pr.geom->lv[0].h;
    vsg_status st;
    const size_t n = (size_t)npairs * cap;
    if ((st = matcher_ensure(m, kSlotOut, n * 12)) || (st = matcher_ensure(m, kSlotAreaQueries, n * 8))) return st;
    int *bd = (int *)m->buf[kSlotOut], *bi = bd + n, *sad = bi + n;
    float *ur = (float *)m->buf[kSlotAreaQueries], *dp = ur + n;
    cudaStream_t s = m->stream;
    const float max_d = mbf / mb;
    const size_t smem = (size_t)cap * sizeof(RightKp);
    if (smem > 200 * 1024) { set_error("vsg_stereo_match_batch: too many keypoints per image (%d)", cap); return VSG_ERR_INVALID; }
    if (smem > 48 * 1024) CK(cudaFuncSetAttribute(stereo_search_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    stereo_search_batch_kernel<<<dim3((cap + 127) / 128, npairs), 128, smem, s>>>(P, pr.kps_dev, (const uint4 *)pr.desc_dev, pr.n_dev,
                                                                                 cap, max_d, bd, bi);
    stereo_sad_batch_kernel<<<dim3((cap + 7) / 8, npairs), 256, 0, s>>>(P, pr.kps_dev, pr.n_dev, cap, bd, bi, max_d, mbf, sad, ur, dp);
    stereo_median_kernel<<<npairs, 256, 0, s>>>(cap, sad, ur, dp);
    count_launch(3);
    CK(cudaGetLastError());
    CK(cudaMemcpy2DAsync(u_right_out, (size_t)capacity * 4, ur, (size_t)cap * 4, (size_t)cap * 4, npairs, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpy2DAsync(depth_out, (size_t)capacity * 4, dp, (size_t)cap * 4, (size_t)cap * 4, npairs, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return VSG_OK;
}
