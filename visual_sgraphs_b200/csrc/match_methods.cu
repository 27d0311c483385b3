// match_methods.cu — the reference's Search* methods on flattened views (single-camera branches).
//
// Reference (snt-arg/visual_sgraphs):
//   Frame::AssignFeaturesToGrid / PosInGrid / GetFeaturesInArea   orb_slam3/src/Frame.cc:521-553, 870-880, 802-868
//   ORBmatcher::SearchByProjection(Frame&, vector<MapPoint*>&)     orb_slam3/src/ORBmatcher.cc:42-144
//   ORBmatcher::SearchByProjection(Frame&, const Frame&)           :1667-1878
//   ORBmatcher::SearchByBoW(KeyFrame*, Frame&)                     :226-428
//   ORBmatcher::SearchForInitialization                            :643-756
//   ORBmatcher::ComputeThreeMaxima + rotation histogram            :2002-2043, idiom :351-358
//
// Split of work: area_search_kernel answers every window query of a call in parallel — the grid walk of
// GetFeaturesInArea (same cell order, same level / distance tests, same float arithmetic) fused with the
// 256-bit Hamming distance of each surviving candidate — and returns per-query candidate lists in the
// reference's order.  The methods' order-dependent bookkeeping (a keypoint claimed by an earlier map point
// is skipped by later ones, vMatchedDistance stealing, the rotation histogram) is sequential by
// definition; it is replayed on the host over those lists, which is O(#candidates) integer work.
#include <algorithm>
#include <chrono>
#include <cstring>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <string>
#include <vector>

#include "match_internal.cuh"
#include "comm_internal.h"

namespace vsg {

__device__ __forceinline__ int hamming256(const uint4 &a0, const uint4 &a1, const uint4 &b0, const uint4 &b1) {
    return __popc(a0.x ^ b0.x) + __popc(a0.y ^ b0.y) + __popc(a0.z ^ b0.z) + __popc(a0.w ^ b0.w) +
           __popc(a1.x ^ b1.x) + __popc(a1.y ^ b1.y) + __popc(a1.z ^ b1.z) + __popc(a1.w ^ b1.w);
}

// One WARP per query (Frame.cc:802-868).  The cells of the query window, flattened in the reference's walk order
// (ix outer, iy inner), are dealt to the lanes 32 at a time; every lane filters the keypoints of its cell (level range,
// |dx|, |dy| < r, the caller's stereo gate) and measures their Hamming distance to the query descriptor.  A warp prefix
// sum over the per-lane hit counts gives every hit its position in the query's list, so the list comes out in exactly
// the order the reference's three nested loops produce.  Two sweeps: the first only counts (the query's segment of the
// output is then reserved with one atomic), the second stores.
__global__ void __launch_bounds__(256) area_search_kernel(FrameDev f, int nq, const AreaQuery *__restrict__ qs,
                                                          const uint4 *__restrict__ qdesc, int *__restrict__ q_off,
                                                          int *__restrict__ q_cnt, int2 *__restrict__ out, int cap,
                                                          int *__restrict__ total) {
    const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (q >= nq) return;
    const AreaQuery a = qs[q];
    const int min_cx = max(0, (int)floorf((a.x - f.min_x - a.r) * f.inv_w));
    const int max_cx = min(f.cols - 1, (int)ceilf((a.x - f.min_x + a.r) * f.inv_w));
    const int min_cy = max(0, (int)floorf((a.y - f.min_y - a.r) * f.inv_h));
    const int max_cy = min(f.rows - 1, (int)ceilf((a.y - f.min_y + a.r) * f.inv_h));
    const bool ok = !(min_cx >= f.cols || max_cx < 0 || min_cy >= f.rows || max_cy < 0) && a.r == a.r;
    if (!ok) {
        if (lane == 0) { q_off[q] = 0; q_cnt[q] = 0; }
        return;
    }
    const bool check_levels = (a.min_level > 0) || (a.max_level >= 0);
    const int di = a.desc_idx >= 0 ? a.desc_idx : q;
    const uint4 qa = __ldg(qdesc + 2 * di), qb = __ldg(qdesc + 2 * di + 1);
    const int ncy = max_cy - min_cy + 1, ncell = (max_cx - min_cx + 1) * ncy;
    int off = 0, stored = 0;
    for (int pass = 0; pass < 2; ++pass) {
        int before = 0;                                   // hits of the cells ahead of this round
        for (int base = 0; base < ncell; base += 32) {
            const int k = base + lane;
            int jb = 0, je = 0;
            if (k < ncell) {
                const int ix = min_cx + k / ncy, iy = min_cy + k % ncy;
                const int c = ix * f.rows + iy;
                jb = f.cell_ptr[c];
                je = f.cell_ptr[c + 1];
            }
            // sweep 0 counts this lane's hits; sweep 1 needs the count first for the positions, so it filters twice
            int mine = 0;
            for (int rep = 0; rep <= pass; ++rep) {
                int w = 0, pos = 0;
                if (rep == 1) {                           // positions: exclusive prefix of `mine` over the lanes
                    int incl = mine;
#pragma unroll
                    for (int d = 1; d < 32; d <<= 1) {
                        const int v = __shfl_up_sync(0xffffffffu, incl, d);
                        if (lane >= d) incl += v;
                    }
                    pos = off + before + incl - mine;
                    before += __shfl_sync(0xffffffffu, incl, 31);
                }
                for (int j = jb; j < je; ++j) {
                    const int idx = f.cell_idx[j];
                    if (check_levels) {
                        const int o = f.octave[idx];
                        if (o < a.min_level) continue;
                        if (a.max_level >= 0 && o > a.max_level) continue;
                    }
                    const float2 p = f.xy[idx];
                    if (!(fabsf(p.x - a.x) < a.r && fabsf(p.y - a.y) < a.r)) continue;
                    if (a.rr >= 0.f && f.u_right) {
                        const float ur = f.u_right[idx];
                        if (ur > 0 && fabsf(a.xr - ur) > a.rr) continue;
                    }
                    const int d = hamming256(qa, qb, __ldg(f.desc + 2 * idx), __ldg(f.desc + 2 * idx + 1));
                    if (d > a.max_dist) continue;         // farther than the caller can use: not listed
                    if (rep == 1 && pos + w < cap) out[pos + w] = make_int2(idx, d);
                    ++w;
                }
                mine = w;
            }
            if (pass == 0) {
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, d);
                stored += mine;
            }
        }
        if (pass == 0) {
            if (stored == 0) break;
            if (lane == 0) off = atomicAdd(total, stored);
            off = __shfl_sync(0xffffffffu, off, 0);
        }
    }
    if (lane == 0) { q_off[q] = off; q_cnt[q] = stored; }
}

static bool timing_on() { static const bool on = getenv("VSG_TIMING") != nullptr; return on; }
struct PhaseTimer {
    std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
    const char *what;
    explicit PhaseTimer(const char *w) : what(w) {}
    void mark(const char *phase) {
        if (!timing_on()) return;
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[vsg timing] %s: %s %.3f ms\n", what, phase, std::chrono::duration<double, std::milli>(now - t).count());
        t = now;
    }
};

// The same walk, but instead of listing the candidates it keeps each query's BEST one on the device: the smallest Hamming
// distance among the keypoints that pass the window / level gates (and, for the pose-based Fuse, the chi-square reprojection
// gates of ORBmatcher.cc:1273-1299), first candidate in the reference's scan order on ties (its updates are strict '<').
// For the methods whose queries do not depend on one another — the Fuse searches and SearchBySim3 — this is the whole
// search: one launch, one (index, distance) pair per query back to the host.  Called by a whole warp for one query.
template <bool kChi2>
__device__ __forceinline__ int2 window_best(const FrameDev &f, const Chi2Gate &gate, const AreaQuery &a, const uint4 *__restrict__ qdesc,
                                            int di, int lane) {
    const int min_cx = max(0, (int)floorf((a.x - f.min_x - a.r) * f.inv_w));
    const int max_cx = min(f.cols - 1, (int)ceilf((a.x - f.min_x + a.r) * f.inv_w));
    const int min_cy = max(0, (int)floorf((a.y - f.min_y - a.r) * f.inv_h));
    const int max_cy = min(f.rows - 1, (int)ceilf((a.y - f.min_y + a.r) * f.inv_h));
    const bool ok = !(min_cx >= f.cols || max_cx < 0 || min_cy >= f.rows || max_cy < 0) && a.r == a.r;
    int best = INT_MAX, best_idx = -1;
    if (ok) {
        const bool check_levels = (a.min_level > 0) || (a.max_level >= 0);
        const uint4 qa = __ldg(qdesc + 2 * di), qb = __ldg(qdesc + 2 * di + 1);
        const int ncy = max_cy - min_cy + 1, ncell = (max_cx - min_cx + 1) * ncy;
        for (int base = 0; base < ncell; base += 32) {            // cells in the reference's walk order, 32 per round
            const int k = base + lane;
            int jb = 0, je = 0;
            if (k < ncell) {
                const int ix = min_cx + k / ncy, iy = min_cy + k % ncy;
                const int c = ix * f.rows + iy;
                jb = f.cell_ptr[c];
                je = f.cell_ptr[c + 1];
            }
            int mine = INT_MAX, mine_idx = -1;
            for (int j = jb; j < je; ++j) {
                const int idx = f.cell_idx[j];
                const int o = f.octave[idx];
                if (check_levels) {
                    if (o < a.min_level) continue;
                    if (a.max_level >= 0 && o > a.max_level) continue;
                }
                const float2 p = f.xy[idx];
                if (!(fabsf(p.x - a.x) < a.r && fabsf(p.y - a.y) < a.r)) continue;
                if (kChi2) {                                      // :1273-1299 (a.xr carries the projected right coordinate)
                    const float ex = a.x - p.x, ey = a.y - p.y;
                    const float ur = f.u_right ? f.u_right[idx] : -1.f;
                    if (ur >= 0) {
                        const float er = a.xr - ur;
                        const float e2 = ex * ex + ey * ey + er * er;
                        if ((double)(e2 * gate.inv_sigma2[o]) > 7.8) continue;
                    } else {
                        const float e2 = ex * ex + ey * ey;
                        if ((double)(e2 * gate.inv_sigma2[o]) > 5.99) continue;
                    }
                }
                const int d = hamming256(qa, qb, __ldg(f.desc + 2 * idx), __ldg(f.desc + 2 * idx + 1));
                if (d < mine) { mine = d; mine_idx = idx; }
            }
            // the round's winner: smallest distance, lowest lane (= earliest cell) on ties
            unsigned key = mine == INT_MAX ? 0xFFFFFFFFu : ((unsigned)mine << 5) | (unsigned)lane;
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) key = min(key, __shfl_xor_sync(0xffffffffu, key, d));
            if (key != 0xFFFFFFFFu) {
                const int rd = (int)(key >> 5), rl = (int)(key & 31);
                const int ridx = __shfl_sync(0xffffffffu, mine_idx, rl);
                if (rd < best) { best = rd; best_idx = ridx; }    // strict: an earlier round keeps a tie
            }
        }
    }
    return make_int2(best_idx, best);
}

template <bool kChi2>
__global__ void __launch_bounds__(256) window_best_kernel(FrameDev f, int nq, const AreaQuery *__restrict__ qs,
                                                          const uint4 *__restrict__ qdesc, Chi2Gate gate,
                                                          int2 *__restrict__ best_out) {
    const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (q >= nq) return;
    const AreaQuery a = qs[q];
    const int2 r = window_best<kChi2>(f, gate, a, qdesc, a.desc_idx >= 0 ? a.desc_idx : q, lane);
    if (lane == 0) best_out[q] = r;
}

// The same over the queries of several keyframes at once (Fuse into every neighbour of a keyframe): query q searches
// targets[q_target[q]] with that keyframe's own grid, level and chi-square tables, and descriptor row desc_idx.
__global__ void __launch_bounds__(256) window_best_multi_kernel(const FuseTarget *__restrict__ targets, int nq,
                                                                const AreaQuery *__restrict__ qs, const int *__restrict__ q_target,
                                                                const uint4 *__restrict__ qdesc, int2 *__restrict__ best_out) {
    const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (q >= nq) return;
    const AreaQuery a = qs[q];
    const FuseTarget &t = targets[q_target[q]];
    const int2 r = window_best<true>(t.f, t.gate, a, qdesc, a.desc_idx, lane);
    if (lane == 0) best_out[q] = r;
}

static FrameDev frame_dev(const vsg_frame *f) {
    return FrameDev{f->n, f->cols, f->rows, f->min_x, f->min_y, f->inv_w, f->inv_h, f->xy, f->octave,
                    f->has_right ? f->u_right : nullptr, (const uint4 *)f->desc, f->cell_ptr, f->cell_idx};
}

static Chi2Gate chi2_gate(const vsg_frame *f, const float *inv_sigma2) {
    Chi2Gate gate;
    for (int l = 0; l < kMaxLevels; ++l) gate.inv_sigma2[l] = inv_sigma2 && l < f->n_levels ? inv_sigma2[l] : 0.f;
    return gate;
}

// Best candidate of every query (see window_best_kernel); out[k] = (keypoint index or -1, distance or INT_MAX), host memory.
vsg_status area_best(vsg_matcher *m, const vsg_frame *f, int nq, const AreaQuery *qs, const uint8_t *qdesc, const float *inv_sigma2,
                     std::vector<int2> &out) {
    out.assign(nq, make_int2(-1, INT_MAX));
    if (nq == 0) return VSG_OK;
    cudaStream_t s = m->stream;
    vsg_status st;
    if ((st = matcher_ensure(m, kSlotAreaQueries, (size_t)nq * sizeof(AreaQuery))) ||
        (st = matcher_ensure(m, kSlotAreaQdesc, (size_t)nq * 32)) || (st = matcher_ensure(m, kSlotAreaCounts, (size_t)nq * sizeof(int2))) ||
        (st = matcher_ensure_host(m, kHostAreaCounts, (size_t)nq * sizeof(int2))))
        return st;
    AreaQuery *qs_d = (AreaQuery *)m->buf[kSlotAreaQueries];
    uint4 *qdesc_d = (uint4 *)m->buf[kSlotAreaQdesc];
    int2 *best_d = (int2 *)m->buf[kSlotAreaCounts];
    CK(cudaMemcpyAsync(qs_d, qs, (size_t)nq * sizeof(AreaQuery), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(qdesc_d, qdesc, (size_t)nq * 32, cudaMemcpyHostToDevice, s));
    const FrameDev fd = frame_dev(f);
    const Chi2Gate gate = chi2_gate(f, inv_sigma2);
    if (inv_sigma2)
        window_best_kernel<true><<<(nq + 7) / 8, 256, 0, s>>>(fd, nq, qs_d, qdesc_d, gate, best_d);
    else
        window_best_kernel<false><<<(nq + 7) / 8, 256, 0, s>>>(fd, nq, qs_d, qdesc_d, gate, best_d);
    count_launch();
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(m->hbuf[kHostAreaCounts], best_d, (size_t)nq * sizeof(int2), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    memcpy(out.data(), m->hbuf[kHostAreaCounts], (size_t)nq * sizeof(int2));
    return VSG_OK;
}

vsg_status area_best_multi(vsg_matcher *m, int ntargets, const vsg_frame *const *frames, const float *const *inv_sigma2, int nq,
                           const AreaQuery *qs, const int *q_target, int n_qdesc, const uint8_t *qdesc, std::vector<int2> &out) {
    out.assign(nq, make_int2(-1, INT_MAX));
    if (nq == 0) return VSG_OK;
    cudaStream_t s = m->stream;
    vsg_status st;
    // one staging block, one H2D copy: target table, queries, their targets, descriptor rows (16-byte aligned sections)
    const size_t o_tgt = 0, o_q = o_tgt + up16((size_t)ntargets * sizeof(FuseTarget)),
                 o_qt = o_q + up16((size_t)nq * sizeof(AreaQuery)), o_desc = o_qt + up16((size_t)nq * sizeof(int)),
                 total = o_desc + (size_t)n_qdesc * 32;
    if ((st = matcher_ensure(m, kSlotBestMultiIn, total)) || (st = matcher_ensure(m, kSlotBestMultiOut, (size_t)nq * sizeof(int2))) ||
        (st = matcher_ensure_host(m, kHostBestMultiIn, total)) || (st = matcher_ensure_host(m, kHostBestMultiOut, (size_t)nq * sizeof(int2))))
        return st;
    uint8_t *h = (uint8_t *)m->hbuf[kHostBestMultiIn], *d = (uint8_t *)m->buf[kSlotBestMultiIn];
    FuseTarget *ht = (FuseTarget *)(h + o_tgt);
    for (int t = 0; t < ntargets; ++t) ht[t] = FuseTarget{frame_dev(frames[t]), chi2_gate(frames[t], inv_sigma2[t])};
    memcpy(h + o_q, qs, (size_t)nq * sizeof(AreaQuery));
    memcpy(h + o_qt, q_target, (size_t)nq * sizeof(int));
    memcpy(h + o_desc, qdesc, (size_t)n_qdesc * 32);
    CK(cudaMemcpyAsync(d, h, total, cudaMemcpyHostToDevice, s));
    window_best_multi_kernel<<<(nq + 7) / 8, 256, 0, s>>>((const FuseTarget *)(d + o_tgt), nq, (const AreaQuery *)(d + o_q),
                                                          (const int *)(d + o_qt), (const uint4 *)(d + o_desc),
                                                          (int2 *)m->buf[kSlotBestMultiOut]);
    count_launch();
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(m->hbuf[kHostBestMultiOut], m->buf[kSlotBestMultiOut], (size_t)nq * sizeof(int2), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    memcpy(out.data(), m->hbuf[kHostBestMultiOut], (size_t)nq * sizeof(int2));
    return VSG_OK;
}

// The window search both list forms share: uploads the queries and n_qdesc descriptor rows, launches area_search_kernel with
// room for init_cap entries (or more if the slot already has it) and, if the lists overflow that, once more with room for all
// of them.  The lists stay on the device (kSlotAreaCounts: off[nq], cnt[nq], total; kSlotAreaRaw: the entries); host slot
// kHostAreaCounts (host_ints ints) receives off, cnt and total if with_offsets, else the total alone.
static vsg_status area_search_launch(vsg_matcher *m, const vsg_frame *f, int nq, const AreaQuery *qs, const uint8_t *qdesc,
                                     int n_qdesc, size_t init_cap, bool with_offsets, size_t host_ints, PhaseTimer &pt, int *total) {
    cudaStream_t s = m->stream;
    vsg_status st;
    if ((st = matcher_ensure(m, kSlotAreaQueries, (size_t)nq * sizeof(AreaQuery))) ||
        (st = matcher_ensure(m, kSlotAreaQdesc, (size_t)n_qdesc * 32)) ||
        (st = matcher_ensure(m, kSlotAreaCounts, (size_t)(2 * nq + 1) * sizeof(int))) ||
        (st = matcher_ensure_host(m, kHostAreaCounts, host_ints * sizeof(int))))
        return st;
    CK(cudaMemcpyAsync(m->buf[kSlotAreaQueries], qs, (size_t)nq * sizeof(AreaQuery), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(m->buf[kSlotAreaQdesc], qdesc, (size_t)n_qdesc * 32, cudaMemcpyHostToDevice, s));
    int *off_d = (int *)m->buf[kSlotAreaCounts], *total_d = off_d + 2 * nq;
    int *host = (int *)m->hbuf[kHostAreaCounts];
    const FrameDev fd = frame_dev(f);
    size_t cap = std::max<size_t>(m->cap[kSlotAreaRaw] / sizeof(int2), init_cap);
    for (int attempt = 0; attempt < 2; ++attempt) {
        if ((st = matcher_ensure(m, kSlotAreaRaw, cap * sizeof(int2)))) return st;
        CK(cudaMemsetAsync(total_d, 0, sizeof(int), s));
        area_search_kernel<<<(nq + 7) / 8, 256, 0, s>>>(fd, nq, (const AreaQuery *)m->buf[kSlotAreaQueries],
                                                       (const uint4 *)m->buf[kSlotAreaQdesc], off_d, off_d + nq,
                                                       (int2 *)m->buf[kSlotAreaRaw], (int)cap, total_d);
        count_launch();
        if (with_offsets)
            CK(cudaMemcpyAsync(host, off_d, (size_t)(2 * nq + 1) * sizeof(int), cudaMemcpyDeviceToHost, s));
        else
            CK(cudaMemcpyAsync(host, total_d, sizeof(int), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        pt.mark(with_offsets ? "H2D + kernel + D2H of offsets" : "H2D + kernel + D2H of the total");
        *total = host[with_offsets ? 2 * nq : 0];
        if ((size_t)*total <= cap) return VSG_OK;
        cap = (size_t)*total + 1024;             // retry once with the exact size
    }
    set_error("area_search: candidate buffer overflow");
    return VSG_ERR_CAPACITY;
}

vsg_status area_search_raw(vsg_matcher *m, const vsg_frame *f, int nq, const AreaQuery *qs, const uint8_t *qdesc,
                           int n_qdesc, AreaLists *out) {
    PhaseTimer pt("area_search");
    *out = AreaLists();
    if (nq == 0) return VSG_OK;
    int total;
    vsg_status st = area_search_launch(m, f, nq, qs, qdesc, n_qdesc, (size_t)nq * 32, true, (size_t)(2 * nq + 1), pt, &total);
    if (st != VSG_OK || (st = matcher_ensure_host(m, kHostAreaEnt, (size_t)std::max(total, 1) * sizeof(int2)))) return st;
    if (total) {
        CK(cudaMemcpyAsync(m->hbuf[kHostAreaEnt], m->buf[kSlotAreaRaw], (size_t)total * sizeof(int2), cudaMemcpyDeviceToHost,
                           m->stream));
        CK(cudaStreamSynchronize(m->stream));
    }
    pt.mark("D2H of entries");
    const int *host = (const int *)m->hbuf[kHostAreaCounts];
    out->raw = (const int2 *)m->hbuf[kHostAreaEnt];
    out->off = host;
    out->cnt = host + nq;
    return VSG_OK;
}

// Exclusive prefix sum of the per-query counts by one CTA (tiles of 1024 with a running carry): ptr[q] = position of query
// q's list in query order, ptr[n] = number of entries.
__global__ void __launch_bounds__(1024) scan_counts_kernel(const int *__restrict__ cnt, int n, int *__restrict__ ptr) {
    __shared__ int s_warp[32];
    __shared__ int s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < n; base += 1024) {
        const int i = base + tid;
        const int v = i < n ? cnt[i] : 0;
        int incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int x = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += x;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        int wsum = lane < 32 ? s_warp[lane] : 0, wincl = wsum;   // every warp scans the 32 warp totals
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int x = __shfl_up_sync(0xffffffffu, wincl, d);
            if (lane >= d) wincl += x;
        }
        const int warp_before = __shfl_sync(0xffffffffu, wincl - wsum, warp);
        const int tile_total = __shfl_sync(0xffffffffu, wincl, 31);
        const int carry = s_carry;
        if (i < n) ptr[i] = carry + warp_before + incl - v;
        __syncthreads();
        if (tid == 0) s_carry = carry + tile_total;
        __syncthreads();
    }
    if (tid == 0) ptr[n] = s_carry;
}

// Copies every query's segment to its place in query order and tags each entry with its query.
__global__ void __launch_bounds__(256) order_segments_kernel(const int2 *__restrict__ raw, const int *__restrict__ off,
                                                             const int *__restrict__ cnt, const int *__restrict__ ptr, int nq,
                                                             int2 *__restrict__ ent, int *__restrict__ qid) {
    const int q = blockIdx.x * 256 + threadIdx.x;
    if (q >= nq) return;
    const int n = cnt[q], src = off[q], dst = ptr[q];
    for (int c = 0; c < n; ++c) {
        ent[dst + c] = raw[src + c];
        qid[dst + c] = q;
    }
}

// area_search_raw with the lists re-ordered on the device: entries of query 0, then of query 1, ... (each list still in
// the reference's candidate order), ptr[nq + 1], and the query of every entry.  For callers whose replay wants to walk
// ALL entries front to back (a map much larger than the frame: most entries are skipped by a one-byte test).
constexpr int kOrderedReplayMinQueries = 20000;   // below this the two extra kernels cost more than the replay saves
struct OrderedLists {
    const int2 *ent = nullptr;
    const int *qid = nullptr, *ptr = nullptr;
    int total = 0;
};
vsg_status area_search_ordered(vsg_matcher *m, const vsg_frame *f, int nq, const AreaQuery *qs, const uint8_t *qdesc,
                               int n_qdesc, OrderedLists *out) {
    PhaseTimer pt("area_search");
    *out = OrderedLists();
    if (nq == 0) return VSG_OK;
    int total;
    vsg_status st = area_search_launch(m, f, nq, qs, qdesc, n_qdesc, (size_t)nq * 4, false, (size_t)nq + 2, pt, &total);
    if (st != VSG_OK) return st;
    if ((st = matcher_ensure(m, kSlotAreaOrder, ((size_t)nq + 1 + std::max(total, 1)) * sizeof(int))) ||
        (st = matcher_ensure(m, kSlotOut, (size_t)std::max(total, 1) * sizeof(int2))) ||
        (st = matcher_ensure_host(m, kHostAreaEnt, (size_t)std::max(total, 1) * sizeof(int2))) ||
        (st = matcher_ensure_host(m, kHostAreaQid, (size_t)std::max(total, 1) * sizeof(int))))
        return st;
    cudaStream_t s = m->stream;
    const int *off_d = (const int *)m->buf[kSlotAreaCounts], *cnt_d = off_d + nq;
    int *ptr_d = (int *)m->buf[kSlotAreaOrder], *qid_d = ptr_d + nq + 1;
    int *host = (int *)m->hbuf[kHostAreaCounts];
    scan_counts_kernel<<<1, 1024, 0, s>>>(cnt_d, nq, ptr_d);
    order_segments_kernel<<<(nq + 255) / 256, 256, 0, s>>>((const int2 *)m->buf[kSlotAreaRaw], off_d, cnt_d, ptr_d, nq,
                                                           (int2 *)m->buf[kSlotOut], qid_d);
    count_launch(2);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(host, ptr_d, (size_t)(nq + 1) * sizeof(int), cudaMemcpyDeviceToHost, s));
    if (total) {
        CK(cudaMemcpyAsync(m->hbuf[kHostAreaEnt], m->buf[kSlotOut], (size_t)total * sizeof(int2), cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(m->hbuf[kHostAreaQid], qid_d, (size_t)total * sizeof(int), cudaMemcpyDeviceToHost, s));
    }
    CK(cudaStreamSynchronize(s));
    pt.mark("ordering + D2H of the lists");
    out->ent = (const int2 *)m->hbuf[kHostAreaEnt];
    out->qid = (const int *)m->hbuf[kHostAreaQid];
    out->ptr = host;
    out->total = total;
    return VSG_OK;
}

// Runs the area search for nq queries and brings the lists back: ptr[nq+1] and (idx, dist) pairs in query order.
vsg_status area_search(vsg_matcher *m, const vsg_frame *f, int nq, const AreaQuery *qs, const uint8_t *qdesc, int n_qdesc,
                       std::vector<int> &ptr, std::vector<int2> &ent) {
    ptr.assign(nq + 1, 0);
    ent.clear();
    AreaLists L;
    vsg_status st = area_search_raw(m, f, nq, qs, qdesc, n_qdesc, &L);
    if (st != VSG_OK || nq == 0) return st;
    int total = 0;
    for (int q = 0; q < nq; ++q) total += L.cnt[q];
    ent.resize(total);
    int w = 0;
    for (int q = 0; q < nq; ++q) {              // segments were allocated in arbitrary order: re-pack by query
        ptr[q] = w;
        for (int k = 0; k < L.cnt[q]; ++k) ent[w++] = L.raw[L.off[q] + k];
    }
    ptr[nq] = w;
    return VSG_OK;
}

// ORBmatcher::ComputeThreeMaxima (ORBmatcher.cc:2002-2043)
void three_maxima(const std::vector<int> *hist, int L, int &ind1, int &ind2, int &ind3) {
    int max1 = 0, max2 = 0, max3 = 0;
    for (int i = 0; i < L; ++i) {
        const int s = (int)hist[i].size();
        if (s > max1) { max3 = max2; max2 = max1; max1 = s; ind3 = ind2; ind2 = ind1; ind1 = i; }
        else if (s > max2) { max3 = max2; max2 = s; ind3 = ind2; ind2 = i; }
        else if (s > max3) { max3 = s; ind3 = i; }
    }
    if (max2 < 0.1f * (float)max1) { ind2 = -1; ind3 = -1; }
    else if (max3 < 0.1f * (float)max1) { ind3 = -1; }
}

int rot_bin(float a1, float a2) {   // :351-358 — factor is 1/HISTO_LENGTH, C round()
    const float factor = 1.0f / HISTO_LENGTH;
    float rot = a1 - a2;
    if (rot < 0.0) rot += 360.0f;
    int bin = (int)std::round(rot * factor);
    if (bin == HISTO_LENGTH) bin = 0;
    return bin;
}

// The KF-F replay of SearchByBoW (ORBmatcher.cc:256-392) over one walk's distances: frame features matched by an earlier
// keyframe feature skipped (:282-283, :303-304), best / second best per camera (:298-322), TH_LOW and ratio gates (the right
// camera's inside the left one's TH_LOW block with its ratio test disabled, :362-366), rotation histogram.  Returns nmatches.
static int bow_replay_kf_f(const vsg_frame_view *KF, const vsg_frame_view *F, int f_nleft, const FeatVec &fb, const BowSeg *segs,
                           int nseg, const uint16_t *dist, float nnratio, int check_ori, int32_t *matches_f_out) {
    for (int i = 0; i < F->n; ++i) matches_f_out[i] = -1;
    std::vector<int> rot_hist[HISTO_LENGTH];
    int nmatches = 0;
    const int nleft = f_nleft < 0 ? F->n : f_nleft;                  // single camera: every feature is a "left" one
    for (int k = 0; k < nseg; ++k) {
        const BowSeg &sg = segs[k];
        int best1 = 256, best_idx_f = -1, best2 = 256;
        int best1r = 256, best_idx_fr = -1, best2r = 256;
        for (int j = sg.jb; j < sg.je; ++j) {
            const int real_f = fb.idx[j];
            if (matches_f_out[real_f] >= 0) continue;                // :282-283, :303-304
            const int d = dist[sg.off + j - sg.jb];
            if (real_f < nleft) {
                if (d < best1) { best2 = best1; best1 = d; best_idx_f = real_f; }
                else if (d < best2) best2 = d;
            } else {
                if (d < best1r) { best2r = best1r; best1r = d; best_idx_fr = real_f; }
                else if (d < best2r) best2r = d;
            }
        }
        if (best1 <= TH_LOW) {
            if (static_cast<float>(best1) < nnratio * static_cast<float>(best2)) {
                matches_f_out[best_idx_f] = sg.i1;
                if (check_ori) rot_hist[rot_bin(KF->keys[sg.i1].angle, F->keys[best_idx_f].angle)].push_back(best_idx_f);
                ++nmatches;
            }
            if (best1r <= TH_LOW) {                                  // ratio test `|| true` (:366)
                matches_f_out[best_idx_fr] = sg.i1;
                if (check_ori) rot_hist[rot_bin(KF->keys[sg.i1].angle, F->keys[best_idx_fr].angle)].push_back(best_idx_fr);
                ++nmatches;
            }
        }
    }
    if (check_ori) apply_rot_filter(rot_hist, [&](int idx) { matches_f_out[idx] = -1; --nmatches; });
    return nmatches;
}

// The window query of map point i (:60-74; the right camera's :146-151): RadiusByViewingCos (:218-224), times th unless th == 1, times the scale
// of the predicted level; levels [level - 1, level]; descriptor row i.  `side` names the camera in the error message.
static vsg_status map_point_query(const vsg_frame *F, const vsg_track_point &mp, int i, float th, float xr, int max_dist,
                                  const char *side, AreaQuery *q) {
    if (mp.level < 0 || mp.level >= (int)F->scale.size()) {
        set_error("map point %d: %slevel %d out of range", i, side, mp.level);
        return VSG_ERR_INVALID;
    }
    float r = (mp.view_cos > 0.998) ? 2.5f : 4.0f;
    if (th != 1.0) r *= th;
    const float win = r * F->scale[mp.level];
    *q = AreaQuery{mp.proj_x, mp.proj_y, win, mp.level - 1, mp.level, xr, win, max_dist, i};
    return VSG_OK;
}

// :48-74 for a single-camera frame: the queries of the map points that reach GetFeaturesInArea into qs and their map point
// indices into q_mp (room for n_mp each), their number into *nq
static vsg_status map_queries(const vsg_frame *F, int n_mp, const vsg_track_point *pts, float th, int far_points, float th_far,
                              int max_dist, AreaQuery *qs, int *q_mp, int *nq) {
    int k = 0;
    for (int i = 0; i < n_mp; ++i) {
        const vsg_track_point &mp = pts[i];
        if (!mp.in_view) continue;
        if (far_points && mp.depth > th_far) continue;
        if (mp.bad) continue;
        const vsg_status st = map_point_query(F, mp, i, th, mp.proj_xr, max_dist, "", qs + k);
        if (st != VSG_OK) return st;
        q_mp[k++] = i;
    }
    *nq = k;
    return VSG_OK;
}

// The best / second-best-by-level scan of :76-141 over one map point's n candidates, cand(c) = (keypoint, distance), skipping
// the blocked keypoints: whether the map point matches, and the keypoint it would take in *best_idx.
enum class MapScan { NoCandidate, RatioRejected, Match };   // none <= TH_HIGH (:123); the `continue` of :124-125; a match
template <class Cand>
static MapScan map_scan(int n, Cand cand, const uint8_t *blocked, const vsg_keypoint *keys, float nnratio, int *best_idx) {
    int best = 256, best_level = -1, best2 = 256, best_level2 = -1, idx = -1;
    for (int c = 0; c < n; ++c) {
        const int2 e = cand(c);
        if (blocked[e.x]) continue;
        if (e.y < best) { best2 = best; best = e.y; best_level2 = best_level; best_level = keys[e.x].octave; idx = e.x; }
        else if (e.y < best2) { best_level2 = keys[e.x].octave; best2 = e.y; }
    }
    *best_idx = idx;
    if (best > TH_HIGH) return MapScan::NoCandidate;
    if (best_level == best_level2 && best > nnratio * best2) return MapScan::RatioRejected;
    return MapScan::Match;
}

// ORBmatcher.cc:1667-1878 over the ncam cameras of the current frame Cur[0 .. ncam): the points of the last frame searched in
// camera c around pts[c] (pts[0] carries the point's octave, angle and flags), their descriptors in desc.  With two cameras a
// point's right-camera search (:1785-1852) is skipped when its left window was empty, whose `continue` (:1727-1728) skips it.
static vsg_status projection_last(vsg_matcher *m, int ncam, const vsg_frame *const *Cur, const uint8_t *occupied, int n_last,
                                  const vsg_proj_point *const *pts, const uint8_t *desc, float th, int mode, int check_ori,
                                  int32_t *assign_out, int *nmatches_out) {
    CK(cudaSetDevice(m->device));
    std::vector<AreaQuery> qs[2];
    std::vector<int> q_src;
    for (int i = 0; i < n_last; ++i) {
        const vsg_proj_point &p = pts[0][i];
        if (!p.valid) continue;
        if (p.octave < 0 || p.octave >= (int)Cur[0]->scale.size()) { set_error("point %d: octave %d out of range", i, p.octave); return VSG_ERR_INVALID; }
        const float radius = th * Cur[0]->scale[p.octave];
        int lo, hi;
        if (mode == 1) { lo = p.octave; hi = -1; }                 // forward  (:1719-1720)
        else if (mode == 2) { lo = 0; hi = p.octave; }             // backward (:1721-1722)
        else { lo = p.octave - 1; hi = p.octave + 1; }             // :1723-1724
        for (int cam = 0; cam < ncam; ++cam)
            qs[cam].push_back(AreaQuery{pts[cam][i].u, pts[cam][i].v, radius, lo, hi, ncam == 1 ? p.ur : 0.f, radius});
        q_src.push_back(i);
    }
    const int nq = (int)q_src.size();
    std::vector<uint8_t> qdesc((size_t)nq * 32);
    for (int k = 0; k < nq; ++k) memcpy(&qdesc[(size_t)k * 32], desc + (size_t)q_src[k] * 32, 32);
    std::vector<int> ptr[2];
    std::vector<int2> ent[2];
    int N = 0;
    for (int cam = 0; cam < ncam; ++cam) {
        const vsg_status st = area_search(m, Cur[cam], nq, qs[cam].data(), qdesc.data(), nq, ptr[cam], ent[cam]);
        if (st != VSG_OK) return st;
        N += Cur[cam]->n;
    }
    std::vector<uint8_t> blocked(occupied, occupied + N);
    for (int i = 0; i < N; ++i) assign_out[i] = -1;
    std::vector<int> rot_hist[HISTO_LENGTH];
    int nmatches = 0;
    for (int k = 0; k < nq; ++k) {
        const vsg_proj_point &p = pts[0][q_src[k]];
        if (ncam == 2 && ptr[0][k] == ptr[0][k + 1]) continue;     // vIndices2.empty() -> continue: no right-camera search either
        for (int cam = 0, offset = 0; cam < ncam; offset += Cur[cam]->n, ++cam) {
            const int2 b = nearest_unclaimed(ent[cam].data() + ptr[cam][k], ent[cam].data() + ptr[cam][k + 1], blocked.data() + offset);
            if (b.x <= TH_HIGH) {
                assign_out[b.y + offset] = q_src[k];
                blocked[b.y + offset] = p.blocks;
                ++nmatches;
                if (check_ori) rot_hist[rot_bin(p.angle, Cur[cam]->keys[b.y].angle)].push_back(b.y + offset);
            }
        }
    }
    if (check_ori) apply_rot_filter(rot_hist, [&](int idx) { assign_out[idx] = -2; --nmatches; });
    if (nmatches_out) *nmatches_out = nmatches;
    return VSG_OK;
}

}  // namespace vsg

using namespace vsg;

extern "C" {

vsg_status vsg_frame_create(vsg_matcher *m, const vsg_frame_view *v, vsg_frame **out) {
    if (!m || !v || !out || v->n < 0 || v->grid_cols < 1 || v->grid_rows < 1 || (v->n > 0 && (!v->keys || !v->descriptors)))
        return VSG_ERR_INVALID;
    // the searches index the level tables (scale factors, the Fuse gate's kMaxLevels sigma table) by keypoint octave
    if (v->n_levels > kMaxLevels || (v->n > 0 && v->n_levels < 1)) {
        set_error("vsg_frame_create: %d pyramid levels, %d keypoints (at most %d levels, at least 1 with keypoints)", v->n_levels,
                  v->n, kMaxLevels);
        return VSG_ERR_INVALID;
    }
    for (int i = 0; i < v->n; ++i)
        if (v->keys[i].octave < 0 || v->keys[i].octave >= v->n_levels) {
            set_error("vsg_frame_create: keypoint %d has octave %d outside [0, %d)", i, v->keys[i].octave, v->n_levels);
            return VSG_ERR_INVALID;
        }
    CK(cudaSetDevice(m->device));
    vsg_frame *f = new vsg_frame();
    f->device = m->device; f->n = v->n; f->cols = v->grid_cols; f->rows = v->grid_rows; f->n_levels = v->n_levels;
    f->min_x = v->min_x; f->min_y = v->min_y; f->inv_w = v->grid_inv_w; f->inv_h = v->grid_inv_h;
    f->has_right = v->u_right != nullptr;
    f->keys.assign(v->keys, v->keys + v->n);
    if (v->scale_factors) f->scale.assign(v->scale_factors, v->scale_factors + v->n_levels);
    if (v->u_right) f->u_right_h.assign(v->u_right, v->u_right + v->n);
    // AssignFeaturesToGrid (Frame.cc:521-553): keypoints appended to their cell in index order; PosInGrid uses round()
    const int ncell = f->cols * f->rows;
    std::vector<int> cell_of(v->n, -1), cptr(ncell + 1, 0), cidx;
    for (int i = 0; i < v->n; ++i) {
        const int px = (int)std::round((v->keys[i].x - v->min_x) * v->grid_inv_w);
        const int py = (int)std::round((v->keys[i].y - v->min_y) * v->grid_inv_h);
        if (px < 0 || px >= f->cols || py < 0 || py >= f->rows) continue;
        cell_of[i] = px * f->rows + py;
        ++cptr[cell_of[i] + 1];
    }
    for (int c = 0; c < ncell; ++c) cptr[c + 1] += cptr[c];
    cidx.resize(cptr[ncell]);
    std::vector<int> fill(cptr.begin(), cptr.end() - 1);
    for (int i = 0; i < v->n; ++i)
        if (cell_of[i] >= 0) cidx[fill[cell_of[i]]++] = i;
    // One pinned staging block, one stream-ordered device allocation, one H2D copy (a Search* call of the drop-in
    // classes uploads a frame every time: six cudaMalloc / cudaFree pairs per call cost more than the search itself).
    const size_t n1 = std::max(v->n, 1);
    const size_t o_xy = 0, o_oct = o_xy + up16(n1 * sizeof(float2)), o_ur = o_oct + up16(n1 * sizeof(int)),
                 o_desc = o_ur + up16(n1 * sizeof(float)), o_cptr = o_desc + up16(n1 * 32),
                 o_cidx = o_cptr + up16((size_t)(ncell + 1) * sizeof(int)),
                 total = o_cidx + up16(std::max<size_t>(cidx.size(), 1) * sizeof(int));
    vsg_status st = matcher_ensure_host(m, kHostFrameStaging, total);
    if (st != VSG_OK) { delete f; return st; }
    uint8_t *h = (uint8_t *)m->hbuf[kHostFrameStaging];
    float2 *hxy = (float2 *)(h + o_xy);
    int *hoct = (int *)(h + o_oct);
    for (int i = 0; i < v->n; ++i) { hxy[i] = make_float2(v->keys[i].x, v->keys[i].y); hoct[i] = v->keys[i].octave; }
    if (v->u_right) memcpy(h + o_ur, v->u_right, (size_t)v->n * sizeof(float));
    if (v->n) memcpy(h + o_desc, v->descriptors, (size_t)v->n * 32);
    memcpy(h + o_cptr, cptr.data(), (size_t)(ncell + 1) * sizeof(int));
    if (!cidx.empty()) memcpy(h + o_cidx, cidx.data(), cidx.size() * sizeof(int));
    cudaStream_t s = m->stream;
    bool ok = cuda_ok(cudaMallocAsync(&f->block, total, s), "cudaMallocAsync") &&
              cuda_ok(cudaMemcpyAsync(f->block, h, total, cudaMemcpyHostToDevice, s), "H2D") &&
              cuda_ok(cudaStreamSynchronize(s), "sync");
    if (!ok) { vsg_frame_destroy(f); return VSG_ERR_CUDA; }
    uint8_t *d = (uint8_t *)f->block;
    f->xy = (float2 *)(d + o_xy); f->octave = (int *)(d + o_oct); f->u_right = (float *)(d + o_ur);
    f->desc = d + o_desc; f->cell_ptr = (int *)(d + o_cptr); f->cell_idx = (int *)(d + o_cidx);
    *out = f;
    return VSG_OK;
}

void vsg_frame_destroy(vsg_frame *f) {
    if (!f) return;
    cudaSetDevice(f->device);
    // every search returns only after its kernels have finished, so the block can go back to the pool right away;
    // the frame may outlive the matcher whose stream allocated it, hence the per-thread stream
    if (f->block) cudaFreeAsync(f->block, cudaStreamPerThread);
    delete f;
}

vsg_status vsg_area_search(vsg_matcher *m, const vsg_frame *f, int nq, const float *qx, const float *qy,
                           const float *qr, const int32_t *min_level, const int32_t *max_level,
                           const uint8_t *qdesc, int32_t *cand_ptr, int32_t *cand_idx, int32_t *cand_dist,
                           int capacity, int *total_out) {
    if (!m || !f || nq < 0 || (nq > 0 && (!qx || !qy || !qr || !qdesc || !cand_ptr))) return VSG_ERR_INVALID;
    CK(cudaSetDevice(m->device));
    std::vector<AreaQuery> qs(nq);
    for (int i = 0; i < nq; ++i)
        qs[i] = AreaQuery{qx[i], qy[i], qr[i], min_level ? min_level[i] : -1, max_level ? max_level[i] : -1, 0.f, -1.f};
    std::vector<int> ptr;
    std::vector<int2> ent;
    vsg_status st = area_search(m, f, nq, qs.data(), qdesc, nq, ptr, ent);
    if (st != VSG_OK) return st;
    for (int i = 0; i <= nq; ++i) cand_ptr[i] = ptr[i];
    if (total_out) *total_out = (int)ent.size();
    if ((int)ent.size() > capacity) return VSG_ERR_CAPACITY;
    for (size_t k = 0; k < ent.size(); ++k) {
        if (cand_idx) cand_idx[k] = ent[k].x;
        if (cand_dist) cand_dist[k] = ent[k].y;
    }
    return VSG_OK;
}

// The largest candidate distance the replay of ORBmatcher.cc:76-141 can use.  Candidates at distance d > TH_HIGH with nnratio * d >= TH_HIGH can neither become the best match (:123) nor, as the
// second best, trigger the ratio rejection (:125: best <= TH_HIGH <= nnratio * d), and every candidate that stays is
// closer than every one dropped — so the replay over the pruned lists gives the identical result.
static int projection_map_max_dist(float nnratio) {
    int d = TH_HIGH + 1;
    while (d < 256 && !(nnratio * (float)d >= (float)TH_HIGH)) ++d;
    return d - 1;
}

// GPU half of SearchByProjection(Frame&, vector<MapPoint*>&): candidate lists of every map point
vsg_status vsg_projection_map_candidates(vsg_matcher *m, const vsg_frame *F, int n_mp, const vsg_track_point *pts,
                                         const uint8_t *mp_desc, float th, int far_points, float th_far,
                                         int32_t *cand_ptr, int32_t *cand_idx, int32_t *cand_dist, int capacity,
                                         int *total_out) {
    if (!m || !F || n_mp < 0 || !cand_ptr || (n_mp > 0 && (!pts || !mp_desc))) return VSG_ERR_INVALID;
    CK(cudaSetDevice(m->device));
    std::vector<AreaQuery> qs(std::max(n_mp, 1));
    std::vector<int> q_mp(std::max(n_mp, 1));
    int nq;
    vsg_status st = map_queries(F, n_mp, pts, th, far_points, th_far, 256, qs.data(), q_mp.data(), &nq);   // full lists: the
    if (st != VSG_OK) return st;                                                                     // resolve's nnratio is not known here
    std::vector<int> ptr;
    std::vector<int2> ent;
    if ((st = area_search(m, F, nq, qs.data(), mp_desc, n_mp, ptr, ent)) != VSG_OK) return st;
    if (total_out) *total_out = (int)ent.size();
    // expand to one list per map point
    int q = 0;
    for (int i = 0; i < n_mp; ++i) {
        cand_ptr[i] = q < nq ? ptr[q] : (int)ent.size();
        if (q < nq && q_mp[q] == i) ++q;
    }
    cand_ptr[n_mp] = (int)ent.size();
    if ((int)ent.size() > capacity) return VSG_ERR_CAPACITY;
    for (size_t k = 0; k < ent.size(); ++k) {
        if (cand_idx) cand_idx[k] = ent[k].x;
        if (cand_dist) cand_dist[k] = ent[k].y;
    }
    return VSG_OK;
}

// host half: the order-dependent replay (no device needed; runs on every rank after the all-gather when the map
// points are sharded over GPUs)
vsg_status vsg_projection_map_resolve(const vsg_frame_view *F, const uint8_t *occupied, int n_mp,
                                      const vsg_track_point *pts, const int32_t *cand_ptr, const int32_t *cand_idx,
                                      const int32_t *cand_dist, float nnratio, int32_t *assign_out, int *nmatches_out) {
    if (!F || F->n < 0 || (F->n > 0 && (!occupied || !assign_out))) return VSG_ERR_INVALID;
    std::vector<uint8_t> blocked(occupied, occupied + F->n);
    std::vector<int32_t> assign(F->n, -1);                 // assign_out stays as it was if the call is rejected
    const vsg_status st = vsg_projection_map_resolve_shard(F, blocked.data(), 0, n_mp, pts, cand_ptr, cand_idx, cand_dist, nnratio,
                                                           assign.data(), nmatches_out);
    if (st == VSG_OK) std::copy(assign.begin(), assign.end(), assign_out);
    return st;
}

// ---- SearchByProjection(Frame&, vector<MapPoint*>&) in two halves that the one-call and the sharded entry points share ----
// GPU half: window queries of the map points that reach GetFeaturesInArea (:48-74), candidate lists with distances back
// on the host (pinned staging of the matcher; valid until its next area search).
struct MapSearch {
    int nq = 0;
    const int *q_mp = nullptr;   // query -> map point index (local to the pts array given)
    bool ordered = false;
    AreaLists R;                 // nq < kOrderedReplayMinQueries: lists as the kernel left them
    OrderedLists L;              // otherwise: entries in query order + the query of every entry
};

static vsg_status projection_map_search(vsg_matcher *m, const vsg_frame *F, int n_mp, const vsg_track_point *pts,
                                        const uint8_t *mp_desc, float th, int far_points, float th_far, float nnratio,
                                        MapSearch *out) {
    PhaseTimer pt("search_by_projection_map");
    // query list in the matcher's pinned staging (a 200k-point map is 7 MB of queries: no fresh pages per call, and the
    // upload runs at the PCIe rate instead of the pageable-memory rate)
    vsg_status st = matcher_ensure_host(m, kHostMapQueries, (size_t)std::max(n_mp, 1) * sizeof(AreaQuery));
    if (st != VSG_OK) return st;
    m->scratch.resize(std::max(n_mp, 1));
    AreaQuery *qs = reinterpret_cast<AreaQuery *>(m->hbuf[kHostMapQueries]);
    int nq;
    st = map_queries(F, n_mp, pts, th, far_points, th_far, projection_map_max_dist(nnratio), qs, m->scratch.data(), &nq);
    if (st != VSG_OK) return st;
    pt.mark("queries");
    out->nq = nq;
    out->q_mp = m->scratch.data();
    out->ordered = nq >= kOrderedReplayMinQueries;
    // tracking-sized calls (a local map of a few thousand points): the lists come back as the kernel left them and the
    // replay visits them query by query — two kernels and a copy less than the ordered form
    st = out->ordered ? area_search_ordered(m, F, nq, qs, mp_desc, n_mp, &out->L) : area_search_raw(m, F, nq, qs, mp_desc, n_mp, &out->R);
    pt.mark("area_search total");
    return st;
}

// The first entry from e on whose keypoint is not claimed (total if none).  Out of line on purpose: inlined next to map_scan,
// the loop index is spilled to the stack and every skipped entry of the ordered replay pays a store and a reload.
__attribute__((noinline)) static int first_unclaimed(const int2 *ent, int e, int total, const uint8_t *blocked) {
    while (e < total && blocked[ent[e].x]) ++e;
    return e;
}

// Host half: the sequential replay of :76-141 in map order.  `blocked` (keypoints holding a map point with observations,
// :88-90) is updated in place so that the replay of the NEXT shard of the map can continue from it; assignments are
// written as index_offset + local map point index.  Returns the number of nmatches++ events.
static int projection_map_replay(const vsg_frame *F, uint8_t *blocked, const MapSearch &S, const vsg_track_point *pts,
                                 float nnratio, int index_offset, int32_t *assign_out) {
    const vsg_keypoint *keys = F->keys.data();
    const int *q_mp = S.q_mp;
    int nmatches = 0;
    auto scan = [&](const int2 *c, const int2 *ce, int k) {
        int idx;
        if (map_scan((int)(ce - c), [c](int j) { return c[j]; }, blocked, keys, nnratio, &idx) != MapScan::Match) return;
        assign_out[idx] = index_offset + q_mp[k];
        blocked[idx] = pts[q_mp[k]].blocks;
        ++nmatches;
    };
    if (!S.ordered) {
        for (int k = 0; k < S.nq; ++k) scan(S.R.raw + S.R.off[k], S.R.raw + S.R.off[k] + S.R.cnt[k], k);
        return nmatches;
    }
    // ONE walk over all entries in query order: an entry whose keypoint is already claimed is skipped by a one-byte test —
    // with a map much larger than the frame that is nearly every entry — and only the first unclaimed entry of a query
    // triggers the scan of that query's list.  (Claims only ever appear, so an entry found claimed stays irrelevant.)
    const OrderedLists &L = S.L;
    for (int e = first_unclaimed(L.ent, 0, L.total, blocked); e < L.total; e = first_unclaimed(L.ent, e, L.total, blocked)) {
        const int k = L.qid[e];
        const int2 *c = L.ent + e, *ce = L.ent + L.ptr[k + 1];
        e = L.ptr[k + 1];
        scan(c, ce, k);
    }
    return nmatches;
}

// ORBmatcher.cc:42-144
vsg_status vsg_search_by_projection_map(vsg_matcher *m, const vsg_frame *F, const uint8_t *occupied, int n_mp,
                                        const vsg_track_point *pts, const uint8_t *mp_desc, float th, int far_points,
                                        float th_far, float nnratio, int32_t *assign_out, int *nmatches_out) {
    if (!m || !F || n_mp < 0 || !assign_out || (n_mp > 0 && (!pts || !mp_desc)) || (F->n > 0 && !occupied)) return VSG_ERR_INVALID;
    CK(cudaSetDevice(m->device));
    MapSearch S;
    const vsg_status st = projection_map_search(m, F, n_mp, pts, mp_desc, th, far_points, th_far, nnratio, &S);
    if (st != VSG_OK) return st;
    std::vector<uint8_t> blocked(occupied, occupied + F->n);
    for (int i = 0; i < F->n; ++i) assign_out[i] = -1;
    const int nmatches = projection_map_replay(F, blocked.data(), S, pts, nnratio, 0, assign_out);
    if (nmatches_out) *nmatches_out = nmatches;
    return VSG_OK;
}

// The same with the MAP POINTS sharded over the ranks of a communicator (BASELINE config 3; SURVEY 8e): this rank holds the
// contiguous shard [shard_begin, shard_begin + n_local) of the map; the frame and `occupied` are replicated.  Every rank runs
// the window search of its shard on its own GPU at the same time.  The order-dependent part of the loop needs, per shard, only
// the claim state the earlier shards left (F->n bytes): it travels down the ranks as a token (ncclSend / ncclRecv), each rank
// replays its own lists when the token arrives, and one ncclAllGather of the per-rank assignments (F->n ints + a count per
// rank) gives every rank the result of the one-call method: a later map point overwrites an earlier one's slot exactly as
// `F.mvpMapPoints[bestIdx] = pMP` does (:130), nmatches counts every assignment event.
vsg_status vsg_search_by_projection_map_sharded(vsg_comm *comm, vsg_matcher *m, const vsg_frame *F, const uint8_t *occupied,
                                                int shard_begin, int n_local, const vsg_track_point *pts_local,
                                                const uint8_t *desc_local, float th, int far_points, float th_far, float nnratio,
                                                int32_t *assign_out, int *nmatches_out) {
    if (!comm || !m || !F || n_local < 0 || shard_begin < 0 || !assign_out || (n_local > 0 && (!pts_local || !desc_local)) ||
        (F->n > 0 && !occupied))
        return VSG_ERR_INVALID;
    CK(cudaSetDevice(m->device));
    const int rank = comm_rank(comm), nranks = comm_size(comm), N = F->n;
    MapSearch S;
    vsg_status st = projection_map_search(m, F, n_local, pts_local, desc_local, th, far_points, th_far, nnratio, &S);
    if (st != VSG_OK) return st;
    // device: token (N bytes, padded), my record (N + 1 ints), everyone's records; pinned host mirrors
    const size_t tok_bytes = ((size_t)N + 15) & ~(size_t)15, rec_ints = (size_t)N + 1;
    if ((st = matcher_ensure(m, kSlotMapShardToken, tok_bytes + rec_ints * 4 * (1 + (size_t)nranks) + 64)) ||
        (st = matcher_ensure_host(m, kHostMapShardToken, tok_bytes + rec_ints * 4 * (1 + (size_t)nranks) + 64)))
        return st;
    uint8_t *tok_d = (uint8_t *)m->buf[kSlotMapShardToken], *tok_h = (uint8_t *)m->hbuf[kHostMapShardToken];
    int32_t *rec_d = (int32_t *)(tok_d + tok_bytes), *all_d = rec_d + rec_ints;
    int32_t *rec_h = (int32_t *)(tok_h + tok_bytes), *all_h = rec_h + rec_ints;
    cudaStream_t s = m->stream;
    if (rank == 0) {
        if (N) memcpy(tok_h, occupied, (size_t)N);
    } else {
        if ((st = comm_recv(comm, tok_d, tok_bytes, rank - 1, s)) != VSG_OK) return st;
        CK(cudaMemcpyAsync(tok_h, tok_d, tok_bytes, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
    }
    for (int i = 0; i < N; ++i) rec_h[i] = -1;
    rec_h[N] = projection_map_replay(F, tok_h, S, pts_local, nnratio, shard_begin, rec_h);
    if (rank + 1 < nranks) {
        CK(cudaMemcpyAsync(tok_d, tok_h, tok_bytes, cudaMemcpyHostToDevice, s));
        if ((st = comm_send(comm, tok_d, tok_bytes, rank + 1, s)) != VSG_OK) return st;
    }
    CK(cudaMemcpyAsync(rec_d, rec_h, rec_ints * 4, cudaMemcpyHostToDevice, s));
    if ((st = comm_all_gather(comm, rec_d, all_d, rec_ints * 4, s)) != VSG_OK) return st;
    CK(cudaMemcpyAsync(all_h, all_d, rec_ints * 4 * nranks, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    int nmatches = 0;
    for (int i = 0; i < N; ++i) assign_out[i] = -1;
    for (int r = 0; r < nranks; ++r) {                      // shard order = map order: later shards overwrite
        const int32_t *rec = all_h + (size_t)r * rec_ints;
        for (int i = 0; i < N; ++i)
            if (rec[i] >= 0) assign_out[i] = rec[i];
        nmatches += rec[N];
    }
    if (nmatches_out) *nmatches_out = nmatches;
    return VSG_OK;
}

// Host-only building block of the sharded method for tests without NCCL: replays ONE shard's candidate lists (as
// vsg_projection_map_candidates returns them) from the claim state `blocked` (in / out, F->n bytes); assign_out entries are
// overwritten with shard_begin + local index where this shard assigns, left alone elsewhere.
vsg_status vsg_projection_map_resolve_shard(const vsg_frame_view *F, uint8_t *blocked, int shard_begin, int n_local,
                                            const vsg_track_point *pts_local, const int32_t *cand_ptr, const int32_t *cand_idx,
                                            const int32_t *cand_dist, float nnratio, int32_t *assign_out, int *nmatches_out) {
    if (!F || n_local < 0 || !cand_ptr || (F->n > 0 && (!blocked || !assign_out || !F->keys)) || (n_local > 0 && !pts_local) ||
        (cand_ptr[n_local] > 0 && (!cand_idx || !cand_dist)))
        return VSG_ERR_INVALID;
    // every index a list can reach is checked before anything is written (one flat pass: lists are short)
    int lo = cand_ptr[0], hi = cand_ptr[0];
    for (int k = 1; k <= n_local; ++k) { lo = std::min(lo, cand_ptr[k]); hi = std::max(hi, cand_ptr[k]); }
    if (lo < 0) { set_error("resolve: negative candidate list offset"); return VSG_ERR_INVALID; }
    for (int c = lo; c < hi; ++c)
        if (cand_idx[c] < 0 || cand_idx[c] >= F->n) { set_error("resolve: candidate index out of range"); return VSG_ERR_INVALID; }
    int nmatches = 0;
    for (int k = 0; k < n_local; ++k) {
        const int32_t *ci = cand_idx + cand_ptr[k], *cd = cand_dist + cand_ptr[k];
        int idx;
        if (map_scan(cand_ptr[k + 1] - cand_ptr[k], [ci, cd](int c) { return make_int2(ci[c], cd[c]); }, blocked, F->keys, nnratio,
                     &idx) != MapScan::Match)
            continue;
        assign_out[idx] = shard_begin + k;
        blocked[idx] = pts_local[k].blocks;
        ++nmatches;
    }
    if (nmatches_out) *nmatches_out = nmatches;
    return VSG_OK;
}

// ORBmatcher.cc:42-216 for a two-camera frame (F.Nleft != -1): per map point the left-camera search (:60-144) and the
// right-camera search (:146-213), both window queries on the device, replayed in map order on the host.
vsg_status vsg_search_by_projection_map_2cam(vsg_matcher *m, const vsg_frame *FL, const vsg_frame *FR, const uint8_t *occupied,
                                             const int32_t *left_to_right, const int32_t *right_to_left, int n_mp,
                                             const vsg_track_point *pts_left, const vsg_track_point *pts_right,
                                             const uint8_t *mp_desc, float th, int far_points, float th_far, float nnratio,
                                             int32_t *assign_out, int *nmatches_out) {
    if (!m || !FL || !FR || n_mp < 0 || !assign_out || (n_mp > 0 && (!pts_left || !pts_right || !mp_desc)) ||
        (FL->n + FR->n > 0 && !occupied) || (FL->n > 0 && !left_to_right) || (FR->n > 0 && !right_to_left))
        return VSG_ERR_INVALID;
    if (FL->has_right || FR->has_right) {
        set_error("vsg_search_by_projection_map_2cam: the per-camera frames of a two-camera rig carry no uRight");
        return VSG_ERR_INVALID;
    }
    CK(cudaSetDevice(m->device));
    const int nL = FL->n, N = nL + FR->n;
    const int max_dist = projection_map_max_dist(nnratio);
    // queries of both cameras; q_of[cam][i] = query number of map point i or -1
    std::vector<AreaQuery> qs[2];
    std::vector<int> q_of[2];
    for (int cam = 0; cam < 2; ++cam) q_of[cam].assign(std::max(n_mp, 1), -1);
    for (int i = 0; i < n_mp; ++i) {
        const vsg_track_point &l = pts_left[i], &r = pts_right[i];
        if (!l.in_view && !r.in_view) continue;                                 // :52-53
        if (far_points && l.depth > th_far) continue;                           // :55-56
        if (l.bad) continue;                                                    // :58-59
        AreaQuery q;
        vsg_status st;
        if (l.in_view) {
            if ((st = map_point_query(FL, l, i, th, 0.f, max_dist, "", &q)) != VSG_OK) return st;
            q_of[0][i] = (int)qs[0].size();
            qs[0].push_back(q);
        }
        if (r.in_view && r.level != -1) {                                       // :146-150; no th factor on this side (:151)
            if ((st = map_point_query(FR, r, i, 1.f, 0.f, max_dist, "right ", &q)) != VSG_OK) return st;
            q_of[1][i] = (int)qs[1].size();
            qs[1].push_back(q);
        }
    }
    // the two searches share the matcher's staging: the left lists are copied out before the right search runs
    std::vector<int2> raw_l;
    std::vector<int> off_l, cnt_l;
    AreaLists L;
    vsg_status st;
    if ((st = area_search_raw(m, FL, (int)qs[0].size(), qs[0].data(), mp_desc, n_mp, &L)) != VSG_OK) return st;
    {
        const int nq = (int)qs[0].size();
        off_l.assign(L.off, L.off + nq);
        cnt_l.assign(L.cnt, L.cnt + nq);
        int total = 0;
        for (int k = 0; k < nq; ++k) total = std::max(total, off_l[k] + cnt_l[k]);
        if (total) raw_l.assign(L.raw, L.raw + total);
    }
    AreaLists R;
    if ((st = area_search_raw(m, FR, (int)qs[1].size(), qs[1].data(), mp_desc, n_mp, &R)) != VSG_OK) return st;

    std::vector<uint8_t> blocked(occupied, occupied + N);
    for (int i = 0; i < N; ++i) assign_out[i] = -1;
    int nmatches = 0;
    auto claim = [&](int slot, int mp) { assign_out[slot] = mp; blocked[slot] = pts_left[mp].blocks; };
    for (int i = 0; i < n_mp; ++i) {
        int idx;
        if (q_of[0][i] >= 0) {
            const int2 *c = raw_l.data() + off_l[q_of[0][i]];
            const MapScan r = map_scan(cnt_l[q_of[0][i]], [c](int j) { return c[j]; }, blocked.data(), FL->keys.data(), nnratio, &idx);
            if (r == MapScan::RatioRejected) continue;                          // `continue` at :124-125: no right-camera search
            if (r == MapScan::Match) {
                claim(idx, i);
                if (left_to_right[idx] != -1) { claim(left_to_right[idx] + nL, i); ++nmatches; }   // :131-136
                ++nmatches;
            }
        }
        if (q_of[1][i] < 0) continue;
        const int2 *c = R.raw + R.off[q_of[1][i]];
        if (map_scan(R.cnt[q_of[1][i]], [c](int j) { return c[j]; }, blocked.data() + nL, FR->keys.data(), nnratio, &idx) !=
            MapScan::Match)                                                     // :176-178: the right camera's claims
            continue;
        if (right_to_left[idx] != -1) { claim(right_to_left[idx], i); ++nmatches; }   // :203-208
        claim(idx + nL, i);
        ++nmatches;
    }
    if (nmatches_out) *nmatches_out = nmatches;
    return VSG_OK;
}

// ORBmatcher.cc:1667-1784 and :1856-1878
vsg_status vsg_search_by_projection_last(vsg_matcher *m, const vsg_frame *Cur, const uint8_t *occupied, int n_last,
                                         const vsg_proj_point *pts, const uint8_t *desc, float th, int mode,
                                         int check_ori, int32_t *assign_out, int *nmatches_out) {
    if (!m || !Cur || n_last < 0 || !assign_out || (n_last > 0 && (!pts || !desc)) || (Cur->n > 0 && !occupied)) return VSG_ERR_INVALID;
    return projection_last(m, 1, &Cur, occupied, n_last, &pts, desc, th, mode, check_ori, assign_out, nmatches_out);
}

// ORBmatcher.cc:1667-1878 with a two-camera current frame (CurrentFrame.Nleft != -1): per last-frame point the left-camera
// search (:1709-1784) and — unless the left window was empty — the right-camera search around its projection through mTrl
// (:1785-1852).
vsg_status vsg_search_by_projection_last_2cam(vsg_matcher *m, const vsg_frame *CurL, const vsg_frame *CurR,
                                              const uint8_t *occupied, int n_last, const vsg_proj_point *pts_left,
                                              const vsg_proj_point *pts_right, const uint8_t *desc, float th, int mode,
                                              int check_ori, int32_t *assign_out, int *nmatches_out) {
    if (!m || !CurL || !CurR || n_last < 0 || !assign_out || (n_last > 0 && (!pts_left || !pts_right || !desc)) ||
        (CurL->n + CurR->n > 0 && !occupied))
        return VSG_ERR_INVALID;
    if (CurL->has_right || CurR->has_right) {
        set_error("vsg_search_by_projection_last_2cam: the per-camera frames of a two-camera rig carry no uRight");
        return VSG_ERR_INVALID;
    }
    const vsg_frame *cur[2] = {CurL, CurR};
    const vsg_proj_point *pts[2] = {pts_left, pts_right};
    return projection_last(m, 2, cur, occupied, n_last, pts, desc, th, mode, check_ori, assign_out, nmatches_out);
}

// ORBmatcher.cc:643-756
vsg_status vsg_search_for_initialization(vsg_matcher *m, const vsg_frame_view *F1, const vsg_frame *F2,
                                         float *prev_matched, int window_size, float nnratio, int check_ori,
                                         int32_t *matches12_out, int *nmatches_out) {
    if (!m || !F1 || !F2 || !matches12_out || (F1->n > 0 && (!prev_matched || !F1->keys || !F1->descriptors))) return VSG_ERR_INVALID;
    CK(cudaSetDevice(m->device));
    std::vector<AreaQuery> qs;
    std::vector<int> q_src;
    for (int i1 = 0; i1 < F1->n; ++i1) {
        const int level1 = F1->keys[i1].octave;
        if (level1 > 0) continue;                                   // :659-661
        qs.push_back(AreaQuery{prev_matched[2 * i1], prev_matched[2 * i1 + 1], (float)window_size, level1, level1, 0.f, -1.f});
        q_src.push_back(i1);
    }
    std::vector<uint8_t> qdesc(qs.size() * 32);
    for (size_t k = 0; k < qs.size(); ++k) memcpy(&qdesc[k * 32], F1->descriptors + (size_t)q_src[k] * 32, 32);
    std::vector<int> ptr;
    std::vector<int2> ent;
    vsg_status st = area_search(m, F2, (int)qs.size(), qs.data(), qdesc.data(), (int)qs.size(), ptr, ent);
    if (st != VSG_OK) return st;
    int nmatches = 0;
    for (int i = 0; i < F1->n; ++i) matches12_out[i] = -1;
    std::vector<int> rot_hist[HISTO_LENGTH];
    std::vector<int> matched_distance(F2->n, INT_MAX), matches21(F2->n, -1);
    for (size_t k = 0; k < qs.size(); ++k) {
        const int i1 = q_src[k];
        int best = INT_MAX, best2 = INT_MAX, best_idx2 = -1;
        for (int c = ptr[k]; c < ptr[k + 1]; ++c) {
            const int i2 = ent[c].x, dist = ent[c].y;
            if (matched_distance[i2] <= dist) continue;             // :682-683
            if (dist < best) { best2 = best; best = dist; best_idx2 = i2; }
            else if (dist < best2) best2 = dist;
        }
        if (best <= TH_LOW) {
            if (best < (float)best2 * nnratio) {
                if (matches21[best_idx2] >= 0) { matches12_out[matches21[best_idx2]] = -1; --nmatches; }
                matches12_out[i1] = best_idx2;
                matches21[best_idx2] = i1;
                matched_distance[best_idx2] = best;
                ++nmatches;
                if (check_ori) rot_hist[rot_bin(F1->keys[i1].angle, F2->keys[best_idx2].angle)].push_back(i1);
            }
        }
    }
    if (check_ori)                                                  // a match stolen later is still in its bin
        apply_rot_filter(rot_hist, [&](int i1) { if (matches12_out[i1] >= 0) { matches12_out[i1] = -1; --nmatches; } });
    for (int i1 = 0; i1 < F1->n; ++i1)                              // :748-751
        if (matches12_out[i1] >= 0) {
            prev_matched[2 * i1] = F2->keys[matches12_out[i1]].x;
            prev_matched[2 * i1 + 1] = F2->keys[matches12_out[i1]].y;
        }
    if (nmatches_out) *nmatches_out = nmatches;
    return VSG_OK;
}

// ORBmatcher.cc:226-428
vsg_status vsg_search_by_bow(vsg_matcher *m, const vsg_frame_view *KF, const uint8_t *kf_mp_valid,
                             const vsg_frame_view *F, int kf_nnodes, const int32_t *kf_nodes, const int32_t *kf_ptr,
                             const int32_t *kf_idx, int f_nnodes, const int32_t *f_nodes, const int32_t *f_ptr,
                             const int32_t *f_idx, float nnratio, int check_ori, int32_t *matches_f_out,
                             int *nmatches_out) {
    return vsg_search_by_bow_2cam(m, KF, kf_mp_valid, F, -1, kf_nnodes, kf_nodes, kf_ptr, kf_idx, f_nnodes, f_nodes, f_ptr, f_idx,
                                  nnratio, check_ori, matches_f_out, nmatches_out);
}

// The same with a two-camera frame (F.Nleft = f_nleft != -1): F's features [0, f_nleft) are the left camera's, the rest
// the right camera's; best / second-best are kept per camera (:298-322) and the right-camera match is taken inside the
// left one's `bestDist1 <= TH_LOW` block with its ratio test disabled (`|| true`, :364-366).  f_nleft == -1: single camera.
vsg_status vsg_search_by_bow_2cam(vsg_matcher *m, const vsg_frame_view *KF, const uint8_t *kf_mp_valid,
                                  const vsg_frame_view *F, int f_nleft, int kf_nnodes, const int32_t *kf_nodes,
                                  const int32_t *kf_ptr, const int32_t *kf_idx, int f_nnodes, const int32_t *f_nodes,
                                  const int32_t *f_ptr, const int32_t *f_idx, float nnratio, int check_ori,
                                  int32_t *matches_f_out, int *nmatches_out) {
    if (!m || !KF || !F || !matches_f_out || kf_nnodes < 0 || f_nnodes < 0 || (KF->n > 0 && !kf_mp_valid) || f_nleft < -1 ||
        f_nleft > F->n)
        return VSG_ERR_INVALID;
    CK(cudaSetDevice(m->device));
    // the merge walk over the two FeatureVectors (:248-376): one query per keyframe feature with a usable map
    // point inside a common node; its candidates are the frame features of that node, in vIndicesF order
    const BowWalk w{KF, kf_mp_valid, FeatVec{kf_nnodes, kf_nodes, kf_ptr, kf_idx}, F, FeatVec{f_nnodes, f_nodes, f_ptr, f_idx}};
    std::vector<BowSeg> segs;
    int64_t npairs = 0;
    const uint16_t *dist;
    const vsg_status st = bow_walk_dists(m, w, segs, &npairs, &dist);
    if (st != VSG_OK) return st;
    const int nmatches = bow_replay_kf_f(KF, F, f_nleft, w.b, segs.data(), (int)segs.size(), dist, nnratio, check_ori, matches_f_out);
    if (nmatches_out) *nmatches_out = nmatches;
    return VSG_OK;
}

// vsg_search_by_bow_2cam(KFs[t] against F) for every target in one upload, one launch and one download
vsg_status vsg_search_by_bow_multi(vsg_matcher *m, int ntargets, const vsg_bow_side *const *KFs, const vsg_bow_side *F,
                                   int f_nleft, float nnratio, int check_ori, int32_t *matches_f_out, int *nmatches_out) {
    if (!m || ntargets < 0) {
        set_error("vsg_search_by_bow_multi: %d targets", ntargets);
        return VSG_ERR_INVALID;
    }
    if (ntargets == 0) return VSG_OK;
    const char *why;
    if (!KFs || !nmatches_out || (F && F->view.n > 0 && !matches_f_out)) {
        set_error("vsg_search_by_bow_multi: null target table or output");
        return VSG_ERR_INVALID;
    }
    if ((why = bow_side_problem(F, false))) {
        set_error("vsg_search_by_bow_multi: F: %s", why);
        return VSG_ERR_INVALID;
    }
    if (f_nleft < -1 || f_nleft > F->view.n) {
        set_error("vsg_search_by_bow_multi: f_nleft %d outside [-1, %d]", f_nleft, F->view.n);
        return VSG_ERR_INVALID;
    }
    std::vector<BowWalk> walks;
    std::vector<BowSeg> segs;
    std::vector<int> seg_ptr;
    int64_t npairs = 0;
    vsg_status st = bow_walk_targets(
        "vsg_search_by_bow_multi", ntargets, [&](int t) { return bow_side_problem(KFs[t], true); },
        [&](int t) {
            const vsg_bow_side &a = *KFs[t];
            return BowWalk{&a.view, a.mp_valid, FeatVec{a.nnodes, a.nodes, a.ptr, a.idx}, &F->view,
                           FeatVec{F->nnodes, F->nodes, F->ptr, F->idx}};
        },
        walks, segs, seg_ptr, &npairs);
    if (st != VSG_OK) return st;
    CK(cudaSetDevice(m->device));
    const uint16_t *dist;
    if ((st = bow_dists(m, ntargets, walks.data(), segs, seg_ptr.data(), npairs, &dist)) != VSG_OK) return st;
    for (int t = 0; t < ntargets; ++t)                                               // in target order, as the loop runs
        nmatches_out[t] = bow_replay_kf_f(&KFs[t]->view, &F->view, f_nleft, walks[t].b, segs.data() + seg_ptr[t],
                                          seg_ptr[t + 1] - seg_ptr[t], dist, nnratio, check_ori,
                                          matches_f_out + (size_t)t * F->view.n);
    return VSG_OK;
}

}  // extern "C"
