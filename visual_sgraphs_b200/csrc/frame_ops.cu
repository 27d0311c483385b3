// frame_ops.cu — the per-keypoint steps Frame's constructors run right after the extractor (SURVEY 8f rank 3).
//
// Reference (snt-arg/visual_sgraphs):
//   Frame::UndistortKeyPoints     orb_slam3/src/Frame.cc:891-922   cv::undistortPoints(mat, mat, mK, mDistCoef, cv::Mat(), mK)
//   Frame::ComputeImageBounds     orb_slam3/src/Frame.cc:924-955   the same call on the four image corners
// OpenCV's undistortPoints (un-vendored; its published algorithm, results pinned bit-exact against cv2 4.13 by the tests):
// double arithmetic throughout, five fixed-point iterations of the Brown-Conrady model, P = K re-projection, float
// results.  The library is compiled with --fmad=false, so the device evaluates the same expression tree unfused.
//
// One thread per point.  Two entry points: host arrays in / out (any point list), and the keypoints of an extractor's
// last host-pointer batch where they already lie in device memory (only the undistorted coordinates come back).
#include <algorithm>

#include "vsg_internal.cuh"

namespace vsg {

struct Calib {
    double fx, fy, cx, cy, ifx, ify;
    double k[12];
};

__device__ __forceinline__ float2 undistort_point(const Calib &c, float u_in, float v_in) {
    const double u = u_in, v = v_in;
    double x = (u - c.cx) * c.ifx, y = (v - c.cy) * c.ify;
    const double x0 = x, y0 = y;
    const double *k = c.k;
    for (int j = 0; j < 5; ++j) {
        const double r2 = x * x + y * y;
        const double icdist = (1 + ((k[7] * r2 + k[6]) * r2 + k[5]) * r2) / (1 + ((k[4] * r2 + k[1]) * r2 + k[0]) * r2);
        if (icdist < 0) {
            x = (u - c.cx) * c.ifx;
            y = (v - c.cy) * c.ify;
            break;
        }
        const double dx = 2 * k[2] * x * y + k[3] * (r2 + 2 * x * x) + k[8] * r2 + k[9] * r2 * r2;
        const double dy = k[2] * (r2 + 2 * y * y) + 2 * k[3] * x * y + k[10] * r2 + k[11] * r2 * r2;
        x = (x0 - dx) * icdist;
        y = (y0 - dy) * icdist;
    }
    // RR = P * R with R = I, P = K; the zero products are kept so that signed zeros and the final 1/ww match
    const double xx = c.fx * x + 0. * y + c.cx, yy = 0. * x + c.fy * y + c.cy, ww = 1. / (0. * x + 0. * y + 1.);
    return make_float2((float)(xx * ww), (float)(yy * ww));
}

__global__ void __launch_bounds__(128) undistort_kernel(Calib c, const float2 *__restrict__ in, int n, float2 *__restrict__ out) {
    const int i = blockIdx.x * 128 + threadIdx.x;
    if (i < n) {
        const float2 p = in[i];
        out[i] = undistort_point(c, p.x, p.y);
    }
}

// keypoints of a batch: kps[frame][cap] records, n[frame] of them valid; rows past n[frame] are written as (-1, -1)
__global__ void __launch_bounds__(128) undistort_batch_kernel(Calib c, const vsg_keypoint *__restrict__ kps,
                                                              const int *__restrict__ n, int cap, int identity,
                                                              float2 *__restrict__ out) {
    const int i = blockIdx.x * 128 + threadIdx.x, frame = blockIdx.y;
    if (i >= cap) return;
    float2 r = make_float2(-1.f, -1.f);
    if (i < n[frame]) {
        const vsg_keypoint kp = kps[(size_t)frame * cap + i];
        r = identity ? make_float2(kp.x, kp.y) : undistort_point(c, kp.x, kp.y);
    }
    out[(size_t)frame * cap + i] = r;
}

static bool make_calib(double fx, double fy, double cx, double cy, const double *dist, int dist_n, Calib *c) {
    if (!(fx != 0.0) || !(fy != 0.0) || dist_n < 0 || dist_n > 12 || (dist_n > 0 && !dist)) return false;
    c->fx = fx; c->fy = fy; c->cx = cx; c->cy = cy;
    c->ifx = 1. / fx; c->ify = 1. / fy;
    for (int i = 0; i < 12; ++i) c->k[i] = i < dist_n ? dist[i] : 0.0;
    return true;
}

}  // namespace vsg

using namespace vsg;

extern "C" {

vsg_status vsg_undistort_keypoints(vsg_matcher *m, int n, const float *xy_in, double fx, double fy, double cx, double cy,
                                   const double *dist, int dist_n, float *xy_out) {
    Calib c;
    if (!m || n < 0 || (n > 0 && (!xy_in || !xy_out)) || !make_calib(fx, fy, cx, cy, dist, dist_n, &c)) {
        set_error("vsg_undistort_keypoints: bad arguments (fx, fy != 0; 0 <= dist_n <= 12)");
        return VSG_ERR_INVALID;
    }
    if (n == 0) return VSG_OK;
    if (dist_n == 0 || dist[0] == 0.0) {          // Frame.cc:893-897: mDistCoef.at<float>(0) == 0.0 -> mvKeysUn = mvKeys
        if (xy_out != xy_in) std::copy(xy_in, xy_in + 2 * (size_t)n, xy_out);
        return VSG_OK;
    }
    CK(cudaSetDevice(m->device));
    vsg_status st;
    if ((st = matcher_ensure(m, kSlotOut, (size_t)n * 8)) || (st = matcher_ensure(m, kSlotAreaQueries, (size_t)n * 8))) return st;
    cudaStream_t s = m->stream;
    CK(cudaMemcpyAsync(m->buf[kSlotOut], xy_in, (size_t)n * 8, cudaMemcpyHostToDevice, s));
    undistort_kernel<<<(n + 127) / 128, 128, 0, s>>>(c, (const float2 *)m->buf[kSlotOut], n, (float2 *)m->buf[kSlotAreaQueries]);
    count_launch();
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(xy_out, m->buf[kSlotAreaQueries], (size_t)n * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return VSG_OK;
}

vsg_status vsg_undistort_keypoints_batch(vsg_matcher *m, vsg_extractor *ex, int nframes, double fx, double fy, double cx,
                                         double cy, const double *dist, int dist_n, float *xy_out, int capacity) {
    Calib c;
    if (!m || !ex || nframes < 0 || (nframes > 0 && !xy_out) || !make_calib(fx, fy, cx, cy, dist, dist_n, &c)) {
        set_error("vsg_undistort_keypoints_batch: bad arguments (fx, fy != 0; 0 <= dist_n <= 12)");
        return VSG_ERR_INVALID;
    }
    PyramidRef pr;
    if (!extractor_pyramid(ex, &pr) || !pr.kps_dev || pr.device != m->device || nframes > pr.nframes) {
        set_error("vsg_undistort_keypoints_batch: the extractor's last call must be a host-pointer batch of >= nframes frames "
                  "on the matcher's device");
        return VSG_ERR_INVALID;
    }
    if (capacity < pr.out_cap) {
        set_error("vsg_undistort_keypoints_batch: capacity %d < vsg_extractor_max_keypoints() = %d", capacity, pr.out_cap);
        return VSG_ERR_CAPACITY;
    }
    if (nframes == 0) return VSG_OK;
    const int identity = dist_n == 0 || dist[0] == 0.0;   // Frame.cc:893-897: mvKeysUn = mvKeys
    CK(cudaSetDevice(m->device));
    CK(cudaStreamSynchronize(pr.stream));
    const int cap = pr.out_cap;
    vsg_status st;
    if ((st = matcher_ensure(m, kSlotAreaQueries, (size_t)nframes * cap * 8))) return st;
    cudaStream_t s = m->stream;
    undistort_batch_kernel<<<dim3((cap + 127) / 128, nframes), 128, 0, s>>>(c, pr.kps_dev, pr.n_dev, cap, identity,
                                                                            (float2 *)m->buf[kSlotAreaQueries]);
    count_launch();
    CK(cudaGetLastError());
    CK(cudaMemcpy2DAsync(xy_out, (size_t)capacity * 8, m->buf[kSlotAreaQueries], (size_t)cap * 8, (size_t)cap * 8, nframes,
                         cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return VSG_OK;
}

}  // extern "C"
