// octree.cu — DistributeOctTree on the device, node-for-node, one CTA per (pyramid level, frame).
//
// Reference (snt-arg/visual_sgraphs):
//   ExtractorNode::DivideNode            orb_slam3/src/ORBextractor.cc:482-537
//   compareNodes                         :539-560
//   ORBextractor::DistributeOctTree      :562-785
//
// How the sequential std::list algorithm is restated for a CTA (DESIGN.md §octree):
//   * A node's key set is a pure function of the node's box path: DivideNode sends a key to a child
//     by comparing its coordinates with the box midpoint only.  So keys never move in memory; each
//     key carries the list position of its node (`node_of`) and every pass re-labels it.
//   * One pass of the reference's main loop divides EVERY multi-key node.  All threads histogram
//     their keys into the four children of their node (shared-memory atomics); the list is then
//     rebuilt in parallel exactly as push_front/erase would leave it — block-wide prefix sums over the
//     list give every child its position: children of the i-th divided node, in n1..n4 order, end up
//     in front of everything pushed before them; single-key nodes keep their relative order behind.
//   * The "careful" phase (:696-759) sorts the expandable nodes with the libstdc++ introsort
//     emulation (introsort.cuh — tie order is part of the result; 64-bit packed items; the partition phase
//     on one thread, the final insertion sort as a parallel stable rank sort);
//     how many of them are divided before the quota is reached, and where their children land, is a
//     block-wide prefix sum over the sorted order; the list is then rebuilt the same way.
//   * Final pick per node = highest response, FIRST in the reference's candidate order on ties
//     (:766-782).  Candidate order is cell-row-major, then row-major inside the cell (:811-874), so
//     the tie break is an atomicMax on (response, ~order_key(x, y)).
#include <algorithm>
#include <cstdio>

#include "introsort.cuh"
#include "vsg_internal.cuh"

namespace vsg {

#ifdef VSG_OCTREE_TIMING
#define OT_DECL long long ot_t[8] = {0, 0, 0, 0, 0, 0, 0, 0}; long long ot_last = clock64(); int ot_rounds = 0;
#define OT_MARK(i) do { const long long now = clock64(); ot_t[i] += now - ot_last; ot_last = now; } while (0)
#else
#define OT_DECL
#define OT_MARK(i) do { } while (0)
#endif

constexpr int kInFlight = 8;

struct ONode {
    short x0, y0, x1, y1;  // UL.x, UL.y, UR.x (== BR.x), BR.y (== BL.y), relative to minBorder
    int count;             // vKeys.size(); bNoMore <=> count == 1
};

// Everything a key pass needs to know about a node in one shared-memory word: the split point in the keys' own (absolute
// level) coordinates, x in bits 0-14 and y in bits 16-30 — the layout of a key word x | y << 16 — and, in bit 31, whether
// the node is divided (in the histogram pass: whether it holds more than one key).
constexpr uint32_t kDivided = 0x80000000u;
__device__ __forceinline__ uint32_t split_word(const ONode &n) {
    const int mx = n.x0 + ((n.x1 - n.x0 + 1) >> 1) + kBorderMin, my = n.y0 + ((n.y1 - n.y0 + 1) >> 1) + kBorderMin;
    return (uint32_t)mx | ((uint32_t)my << 16) | (n.count > 1 ? kDivided : 0u);
}
// child of a key (:498-520: x < midpoint -> left, y < midpoint -> top): 0 .. 3 in n1 .. n4 order
__device__ __forceinline__ int quadrant(uint32_t split, uint32_t xy) {
    return ((xy & 0xFFFFu) >= (split & 0x7FFFu) ? 1 : 0) + ((xy >> 16) >= ((split >> 16) & 0x7FFFu) ? 2 : 0);
}

__device__ __forceinline__ ONode child_of(const ONode &n, int q, int count) {
    const int mx = n.x0 + ((n.x1 - n.x0 + 1) >> 1);
    const int my = n.y0 + ((n.y1 - n.y0 + 1) >> 1);
    ONode c;
    c.x0 = (q & 1) ? mx : n.x0;
    c.x1 = (q & 1) ? n.x1 : mx;
    c.y0 = (q & 2) ? my : n.y0;
    c.y1 = (q & 2) ? n.y1 : my;
    c.count = count;
    return c;
}

// Exclusive prefix sums of three per-thread values over the kThreads threads of the CTA (thread order), in place;
// the block totals are returned in ta, tb, tc.  Contains two barriers.
template <int kThreads>
__device__ __forceinline__ void block_scan3(int &a, int &b, int &c, int (*s_warp)[32], int &ta, int &tb, int &tc) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int ia = a, ib = b, ic = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int xa = __shfl_up_sync(0xffffffffu, ia, d), xb = __shfl_up_sync(0xffffffffu, ib, d),
                  xc = __shfl_up_sync(0xffffffffu, ic, d);
        if (lane >= d) { ia += xa; ib += xb; ic += xc; }
    }
    if (lane == 31) { s_warp[0][warp] = ia; s_warp[1][warp] = ib; s_warp[2][warp] = ic; }
    __syncthreads();
    int wa = 0, wb = 0, wc = 0;
    ta = tb = tc = 0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) {
        const int va = s_warp[0][w], vb = s_warp[1][w], vc = s_warp[2][w];
        if (w < warp) { wa += va; wb += vb; wc += vc; }
        ta += va; tb += vb; tc += vc;
    }
    __syncthreads();
    a = wa + ia - a; b = wb + ib - b; c = wc + ic - c;
}

template <int kThreads>
__global__ void __launch_bounds__(kThreads) octree_kernel(FrameGeom g, const Cand *__restrict__ cand,
                                                     const int *__restrict__ cand_count,
                                                     unsigned short *__restrict__ node_of,
                                                     LevelKp *__restrict__ level_kps,
                                                     int *__restrict__ level_kp_count, int cap) {
    extern __shared__ __align__(16) uint8_t smem[];
    ONode *list_a = reinterpret_cast<ONode *>(smem);
    ONode *list_b = list_a + cap;
    int *cc = reinterpret_cast<int *>(list_b + cap);                       // [cap][4] child key counts
    unsigned short *child_pos = reinterpret_cast<unsigned short *>(cc + 4 * cap);  // [cap][4]
    unsigned short *stay_pos = child_pos + 4 * cap;                        // [cap]
    unsigned short *exp_list = stay_pos + cap;                             // [cap] expandable nodes, push order
    unsigned short *push_off = exp_list + cap;                             // [cap] careful phase: children pushed before r
    unsigned short *exp_off = push_off + cap;                              // [cap] expandable children pushed before r
    SortItem *sort_buf = reinterpret_cast<SortItem *>(exp_off + cap);      // [cap] (cap is a multiple of 4: 8-byte aligned)
    uint32_t *split = reinterpret_cast<uint32_t *>(sort_buf + cap);        // [cap] split_word of every node of the list
    __shared__ int s_size, s_nexp, s_state, s_E, s_T, s_X;
    __shared__ int s_scan[3][32];

    pdl_launch_dependents();
    const int level = blockIdx.x, frame = blockIdx.y;
    const LevelGeom &L = g.lv[level];
    const int tid = threadIdx.x;
    pdl_wait();
    const int n = min(cand_count[frame * g.nlevels + level], L.cand_cap);
    const Cand *keys = cand + L.cand_offset + (int64_t)frame * g.cand_total;
    const uint32_t *key_xy = reinterpret_cast<const uint32_t *>(keys);   // word 2k = x | y << 16 of candidate k
    unsigned short *nof = node_of + L.cand_offset + (int64_t)frame * g.cand_total;
    LevelKp *out = level_kps + (int64_t)frame * g.kp_total + L.kp_offset;
    int *out_count = level_kp_count + frame * g.nlevels + level;
    if (n == 0) {
        if (tid == 0) *out_count = 0;
        return;
    }
    const int N = L.quota;
    const int max_y = L.h - 2 * kBorderMin;  // maxBorderY - minBorderY
    OT_DECL

    // ---- roots (:566-593) ----
    ONode *cur = list_a, *nxt = list_b;
    for (int i = tid; i < L.n_ini; i += kThreads) {
        ONode r;
        r.x0 = (short)(int)__fmul_rn(L.h_x, (float)i);
        r.x1 = (short)(int)__fmul_rn(L.h_x, (float)(i + 1));
        r.y0 = 0;
        r.y1 = (short)max_y;
        r.count = 0;
        cur[i] = r;
    }
    __syncthreads();
    // every key goes to root int(x / hX) (:589-592); the per-root counts are warp ballots + one atomic per warp and
    // root (nIni is 1 .. 4 for real images), not one atomic per key on the same counter
    if (L.n_ini == 1) {
        for (int k = tid; k < n; k += kThreads) nof[k] = 0;
        if (tid == 0) cur[0].count = n;
    } else {
        for (int k0 = 0; k0 < n; k0 += kThreads) {
            const int k = k0 + tid;
            int r = -1;
            if (k < n) {
                r = (int)__fdiv_rn((float)((int)(key_xy[2 * k] & 0xFFFF) - kBorderMin), L.h_x);
                nof[k] = (unsigned short)r;
            }
            if (L.n_ini <= 8) {
                for (int j = 0; j < L.n_ini; ++j) {
                    const unsigned mj = __ballot_sync(0xffffffffu, r == j);
                    if ((tid & 31) == 0 && mj) atomicAdd(&cur[j].count, __popc(mj));
                }
            } else if (r >= 0) {
                atomicAdd(&cur[r].count, 1);
            }
        }
    }
    __syncthreads();
    if (tid == 0) {  // drop empty roots, keep order (:597-608)
        int m = 0;
        for (int i = 0; i < L.n_ini; ++i) {
            stay_pos[i] = (unsigned short)m;
            if (cur[i].count > 0) nxt[m++] = cur[i];
        }
        s_size = m;
        s_state = 0;  // 0 = main passes, 1 = careful phase, 2 = finished
    }
    __syncthreads();
    for (int k = tid; k < n; k += kThreads) nof[k] = stay_pos[nof[k]];
    { ONode *t = cur; cur = nxt; nxt = t; }
    __syncthreads();

    OT_MARK(0);
    // ---- subdivision rounds ----
    while (true) {
        const int size = s_size;
        const int state = s_state;
        if (state == 2) break;
        for (int i = tid; i < size * 4; i += kThreads) cc[i] = 0;
        for (int i = tid; i < size; i += kThreads) split[i] = split_word(cur[i]);
        __syncthreads();
        for (int k0 = tid; k0 < n; k0 += kInFlight * kThreads) {   // kInFlight keys per thread in flight (L2 latency)
            int nd[kInFlight];
            uint32_t xy[kInFlight];
#pragma unroll
            for (int u = 0; u < kInFlight; ++u) {
                const int k = k0 + u * kThreads;
                nd[u] = k < n ? nof[k] : -1;
                xy[u] = k < n ? key_xy[2 * k] : 0u;
            }
#pragma unroll
            for (int u = 0; u < kInFlight; ++u) {
                if (nd[u] < 0) continue;
                const uint32_t w = split[nd[u]];
                if (w & kDivided)
                    atomicAdd(&cc[nd[u] * 4 + quadrant(w, xy[u])], 1);
            }
        }
        __syncthreads();
        OT_MARK(1);

        // every thread owns a contiguous chunk of the list so that prefix sums follow list order
        const int chunk = (size + kThreads - 1) / kThreads;
        const int lo = min(tid * chunk, size), hi = min(lo + chunk, size);
        if (state == 0) {
            // main pass (:626-684): every multi-key node is divided, walking the list front to back; children
            // are pushed to the FRONT in n1..n4 order, single-key nodes keep their relative order behind them
            int kids = 0, stays = 0, exps = 0;
            for (int i = lo; i < hi; ++i) {
                if (cur[i].count == 1) { ++stays; continue; }
                for (int q = 0; q < 4; ++q) { kids += cc[i * 4 + q] > 0; exps += cc[i * 4 + q] > 1; }
            }
            int T, S, X;
            block_scan3<kThreads>(kids, stays, exps, s_scan, T, S, X);     // in: my sums, out: exclusive prefixes; totals in T,S,X
            int push = kids, stay = stays, nexp = exps;
            for (int i = lo; i < hi; ++i) {
                if (cur[i].count == 1) {
                    const int pos = T + stay++;
                    nxt[pos] = cur[i];
                    stay_pos[i] = (unsigned short)pos;
                } else {                                   // divided: split[i] already carries kDivided (count > 1)
                    for (int q = 0; q < 4; ++q) {
                        const int c = cc[i * 4 + q];
                        if (c == 0) continue;
                        const int pos = T - 1 - push++;
                        nxt[pos] = child_of(cur[i], q, c);
                        child_pos[i * 4 + q] = (unsigned short)pos;
                        if (c > 1) exp_list[nexp++] = (unsigned short)pos;
                    }
                }
            }
            if (tid == 0) {
                const int new_size = T + S;
                if (new_size >= N || new_size == size) s_state = 2;           // :690-694
                else if (new_size + X * 3 > N) s_state = 1;                   // :696
                s_size = new_size;
                s_nexp = X;
            }
        } else {
            // careful round (:698-759): sort the expandable nodes, divide from the back until size >= N
            const int m = s_nexp;
            for (int j = tid; j < m; j += kThreads) {
                const int pos = exp_list[j];
                sort_buf[j] = make_sort_item(cur[pos].count, cur[pos].x0, pos);
            }
            for (int i = tid; i < size; i += kThreads) split[i] &= ~kDivided;   // from here on: divided in THIS round
            if (tid == 0) s_E = m;
            __syncthreads();
            OT_MARK(2);
            // std::sort in its two halves (introsort.cuh): the partition phase on one thread, then the final insertion
            // sort — a stable sort of what the partitions left — as one rank computation per element by the whole CTA
            // (child_pos is free until this round's rebuild and serves as the second buffer)
            if (tid == 0) introsort_loop(sort_buf, m);
            __syncthreads();
            {
                SortItem *ranked = reinterpret_cast<SortItem *>(child_pos);
                for (int j = tid; j < m; j += kThreads) ranked[stable_rank(sort_buf, m, j)] = sort_buf[j];
                __syncthreads();
                for (int j = tid; j < m; j += kThreads) sort_buf[j] = ranked[j];
            }
            __syncthreads();
            // processing order r = 0 .. m-1 is sort_buf[m-1-r] (:709 walks the sorted vector from the back).  Node r
            // contributes c_r non-empty children (e_r of them expandable); the list has size + sum_{i<=r}(c_i - 1)
            // nodes after it, and the walk stops after the first r where that reaches N (:753-754).  c_r >= 1, so
            // the running size is monotone: the stop index is a block-wide minimum, the landing positions of the
            // children are exclusive prefix sums over r.
            const int mchunk = (m + kThreads - 1) / kThreads;
            const int rlo = min(tid * mchunk, m), rhi = min(rlo + mchunk, m);
            int csum = 0, esum = 0, zero = 0;
            for (int r = rlo; r < rhi; ++r) {
                const int pos = sort_item_ref(sort_buf[m - 1 - r]);
                for (int q = 0; q < 4; ++q) { csum += cc[pos * 4 + q] > 0; esum += cc[pos * 4 + q] > 1; }
            }
            int Tall, Xall, Zall;
            block_scan3<kThreads>(csum, esum, zero, s_scan, Tall, Xall, Zall);   // csum / esum are now exclusive prefixes
            {
                int run_c = csum, run_e = esum;
                for (int r = rlo; r < rhi; ++r) {
                    const int pos = sort_item_ref(sort_buf[m - 1 - r]);
                    push_off[r] = (unsigned short)run_c;
                    exp_off[r] = (unsigned short)run_e;
                    for (int q = 0; q < 4; ++q) { run_c += cc[pos * 4 + q] > 0; run_e += cc[pos * 4 + q] > 1; }
                    if (size + run_c - (r + 1) >= N) { atomicMin(&s_E, r + 1); break; }
                }
            }
            __syncthreads();
            const int E = s_E;
            // totals over the E divided nodes: the prefix at r = E, recomputed by the one thread whose chunk holds r = E
            // (it may have stopped before reaching it), or the block totals when every node is divided
            if (E == m) {
                if (tid == 0) { s_T = Tall; s_X = Xall; }
            } else if (E >= rlo && E < rhi) {
                int run_c = csum, run_e = esum;
                for (int r = rlo; r < E; ++r) {
                    const int pos = sort_item_ref(sort_buf[m - 1 - r]);
                    for (int q = 0; q < 4; ++q) { run_c += cc[pos * 4 + q] > 0; run_e += cc[pos * 4 + q] > 1; }
                }
                s_T = run_c; s_X = run_e;
            }
            __syncthreads();
            OT_MARK(3);
            const int T = s_T;
            for (int r = tid; r < E; r += kThreads) {
                const int pos = sort_item_ref(sort_buf[m - 1 - r]);
                split[pos] |= kDivided;
                int push = push_off[r], nexp = exp_off[r];
                for (int q = 0; q < 4; ++q) {
                    const int c = cc[pos * 4 + q];
                    if (c == 0) continue;
                    const int np = T - 1 - push++;
                    nxt[np] = child_of(cur[pos], q, c);
                    child_pos[pos * 4 + q] = (unsigned short)np;
                    if (c > 1) exp_list[nexp++] = (unsigned short)np;      // old entries were copied to sort_buf
                }
            }
            __syncthreads();
            int stays = 0;
            for (int i = lo; i < hi; ++i) stays += (split[i] & kDivided) ? 0 : 1;
            int d0 = 0, d1 = 0, S, D0, D1;
            block_scan3<kThreads>(stays, d0, d1, s_scan, S, D0, D1);
            int stay = stays;
            for (int i = lo; i < hi; ++i) {
                if (split[i] & kDivided) continue;
                const int np = T + stay++;
                nxt[np] = cur[i];
                stay_pos[i] = (unsigned short)np;
            }
            if (tid == 0) {
                const int new_size = T + S;
                if (new_size >= N || new_size == size) s_state = 2;           // :753-757
                s_size = new_size;
                s_nexp = s_X;
            }
        }
        __syncthreads();
        OT_MARK(4);
        for (int k0 = tid; k0 < n; k0 += kInFlight * kThreads) {
            int nd[kInFlight];
            uint32_t xy[kInFlight];
#pragma unroll
            for (int u = 0; u < kInFlight; ++u) {
                const int k = k0 + u * kThreads;
                nd[u] = k < n ? nof[k] : -1;
                xy[u] = k < n ? key_xy[2 * k] : 0u;
            }
#pragma unroll
            for (int u = 0; u < kInFlight; ++u) {
                if (nd[u] < 0) continue;
                const int k = k0 + u * kThreads;
                const uint32_t w = split[nd[u]];
                if (w & kDivided)
                    nof[k] = child_pos[nd[u] * 4 + quadrant(w, xy[u])];
                else
                    nof[k] = stay_pos[nd[u]];
            }
        }
        { ONode *t = cur; cur = nxt; nxt = t; }
        __syncthreads();
        OT_MARK(5);
#ifdef VSG_OCTREE_TIMING
        ++ot_rounds;
#endif
    }

    // ---- best key per node (:766-782): highest response, first in the reference's candidate order on ties ----
    // two passes of native 32-bit shared-memory atomics: the maximum response per node, then the smallest order key
    // among the keys that carry it
    const int size = s_size;
    unsigned *best_score = reinterpret_cast<unsigned *>(cc);            // [size]  (cc is free once the tree is final)
    unsigned *best_order = best_score + cap;                            // [size]
    for (int i = tid; i < size; i += kThreads) { best_score[i] = 0u; best_order[i] = 0xFFFFFFFFu; }
    __syncthreads();
    for (int k = tid; k < n; k += kThreads) atomicMax(&best_score[nof[k]], (unsigned)keys[k].score + 1u);
    __syncthreads();
    for (int k = tid; k < n; k += kThreads) {
        const Cand c = keys[k];                                // independent iterations: the loads pipeline
        const int node = nof[k];
        if ((unsigned)c.score + 1u != best_score[node]) continue;
        const int rx = c.x - kEdge, ry = c.y - kEdge;          // offset inside the FAST-able area
        const int cx = (int)__umulhi((uint32_t)rx, L.wcell_rcp), cy = (int)__umulhi((uint32_t)ry, L.hcell_rcp);   // rx / w_cell, ry / h_cell
        const unsigned order = ((unsigned)(cy * L.n_cols + cx) << 14) | ((unsigned)(ry - cy * L.h_cell) << 7) |
                               (unsigned)(rx - cx * L.w_cell);
        atomicMin(&best_order[node], order);
    }
    __syncthreads();
    for (int i = tid; i < size && i < L.kp_cap; i += kThreads) {
        const unsigned order = best_order[i];
        const int cell = order >> 14, ly = (order >> 7) & 127, lx = order & 127;
        const int cy = cell / L.n_cols, cx = cell - cy * L.n_cols;
        LevelKp kp;
        kp.x = (unsigned short)(kEdge + cx * L.w_cell + lx);
        kp.y = (unsigned short)(kEdge + cy * L.h_cell + ly);
        kp.score = (unsigned short)(best_score[i] - 1u);
        kp.pad = 0;
        out[i] = kp;
    }
    if (tid == 0) *out_count = min(size, L.kp_cap);
    OT_MARK(6);
#ifdef VSG_OCTREE_TIMING
    if (tid == 0 && frame == 0)
        printf("octree level %d n %d rounds %d: roots %lld | passA %lld | careful-prep %lld | sort+scan %lld | rebuild %lld | passB %lld | best %lld cycles\n",
               level, n, ot_rounds, ot_t[0], ot_t[1], ot_t[2], ot_t[3], ot_t[4], ot_t[5], ot_t[6]);
#endif
}

static int octree_cap(int max_nodes) { return (max_nodes + 3) & ~3; }

size_t octree_smem_bytes(int max_nodes) {
    // list_a, list_b (12 B each), cc (16 B), child_pos (8 B), stay_pos, exp_list, push_off, exp_off (2 B each),
    // sort_buf (8 B), split (4 B)
    return (size_t)octree_cap(max_nodes) * (12 + 12 + 16 + 8 + 2 + 2 + 2 + 2 + 8 + 4) + 64;
}

vsg_status octree_static_smem_bytes(size_t *bytes) {
    cudaFuncAttributes a256, a512;
    CK(cudaFuncGetAttributes(&a256, octree_kernel<256>));
    CK(cudaFuncGetAttributes(&a512, octree_kernel<512>));
    *bytes = std::max(a256.sharedSizeBytes, a512.sharedSizeBytes);
    return VSG_OK;
}

vsg_status launch_octree(const FrameGeom &g, const Cand *cand, const int *cand_count, unsigned short *node_of,
                         LevelKp *level_kps, int *level_kp_count, int max_nodes, int nframes, cudaStream_t s) {
    const int cap = octree_cap(max_nodes);
    const size_t smem = octree_smem_bytes(max_nodes);
    // A few frames: one CTA per SM at most, and a CTA of 8 warps leaves three quarters of the SM's issue slots empty while it
    // walks its keys — 16 warps: 51 -> 44 us for one 640x480 frame (24 warps: 46, 32 warps: the block-wide scans and barriers
    // cost more than the key passes gain).  Large batches fill the SMs with several 8-warp CTAs instead.
    if (nframes <= 8) {
        if (smem > 48 * 1024)
            CK(cudaFuncSetAttribute(octree_kernel<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CK(launch_kernel(octree_kernel<512>, dim3(g.nlevels, nframes), dim3(512), smem, s, true, g, cand, cand_count, node_of,
                         level_kps, level_kp_count, cap));
    } else {
        if (smem > 48 * 1024)
            CK(cudaFuncSetAttribute(octree_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CK(launch_kernel(octree_kernel<256>, dim3(g.nlevels, nframes), dim3(256), smem, s, true, g, cand, cand_count, node_of,
                         level_kps, level_kp_count, cap));
    }
    count_launch();
    return VSG_OK;
}

}  // namespace vsg
