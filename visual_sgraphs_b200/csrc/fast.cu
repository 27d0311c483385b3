// fast.cu — per-cell FAST-9/16 with cell-local non-max suppression and the iniThFAST/minThFAST retry.
//
// Reference (snt-arg/visual_sgraphs):
//   ORBextractor::ComputeKeyPointsOctTree, cell loop      orb_slam3/src/ORBextractor.cc:811-876
//     cv::FAST(cell, kps, iniThFAST, true); if empty -> cv::FAST(cell, kps, minThFAST, true)   (:832-851)
//   cv::FAST = FAST-9/16 + 3x3 NMS on the cell sub-image (SURVEY Appendix A6):
//     corner at threshold t  <=>  strength K > t, where K = max over the sixteen 9-arcs of the
//     smallest same-signed difference on the arc; response = K - 1; a corner survives NMS iff its
//     response is strictly greater than the responses of its 8 neighbours, where non-corners and
//     pixels outside the cell's interior ([3,w-3) x [3,h-3)) count as 0.
//
// One CTA per (cell, frame).  The cell window is loaded straight into a pair-interleaved shared-memory layout
// (see below), the strength K of every interior pixel is computed once (it does not depend on the threshold),
// NMS runs at iniThFAST and — only if the cell produced nothing — again at minThFAST, exactly the reference's
// retry rule.  Survivors are compacted with warp ballots and appended to the (frame, level) candidate list with
// one global atomic per CTA.  The list order is not the reference's cell-row-major order; the oct-tree only
// depends on order through the first-max-wins tie break, which octree.cu reproduces from the coordinates
// (see order_key there).
#include "blur_device.cuh"
#include "vsg_internal.cuh"

namespace vsg {

// Packed arithmetic: every thread scores TWO pixels of a row at once, lane 0 = interior column j, lane 1 =
// column j + S (S = half the interior width), as 16-bit lanes of one 32-bit register.  sm_100a has native
// two- and three-input packed min/max (VIMNMX.U16x2 / VIMNMX3.U16x2), so the sliding-window minima/maxima of
// the 16-pixel ring cost half the instructions per pixel.  The cell window is re-laid out in shared memory as
// such pairs (T2) so that one aligned 32-bit load fetches a ring position for both pixels.
__device__ __forceinline__ uint32_t min2(uint32_t a, uint32_t b) { uint32_t d; asm("min.u16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b)); return d; }
__device__ __forceinline__ uint32_t max2(uint32_t a, uint32_t b) { uint32_t d; asm("max.u16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b)); return d; }
__device__ __forceinline__ uint32_t min3(uint32_t a, uint32_t b, uint32_t c) { return min2(min2(a, b), c); }   // fused to VIMNMX3
__device__ __forceinline__ uint32_t max3(uint32_t a, uint32_t b, uint32_t c) { return max2(max2(a, b), c); }

constexpr int kFastThreads = 160;
#ifndef VSG_FAST_MINB
#define VSG_FAST_MINB 6   // resident CTAs per SM the register budget is sized for (6 x 160 threads, 64 registers)
#endif
// Row pitches of the two shared-memory planes, in words.  Thread t of the CTA owns pair column j = t % S of row t / S, so a
// warp's 32 consecutive pairs p = row * S + j sit at word row * pitch + j + const = p + row * (pitch - S) + const: with
// pitch = S + 32 every ring / neighbour read of a warp is bank-conflict free.  S = 20 for every full cell of the usual
// 35..40-pixel grids, so the pitch is the constant 52 (a run-time pitch costs more address arithmetic than the conflicts);
// other S only see two-way conflicts on a few lanes.  Minimum sizes: 3 (alignment) + S + 6 halo columns rounded to 4 for
// the pixel pairs, S + 2 for the strengths.
constexpr int kT2Pitch = 52;
constexpr int kS2Pitch = 52;
constexpr int kMaxS = 28;

// The 16-pixel Bresenham ring in OpenCV's order (SURVEY A6): (0,3)(1,3)(2,2)(3,1)(3,0)(3,-1)(2,-2)(1,-3)(0,-3)
// (-1,-3)(-2,-2)(-3,-1)(-3,0)(-3,1)(-2,2)(-1,3).  Strength K of both pixels of the pair at c: max over the 16
// circular 9-windows of the window minimum (bright arcs) / of the negated window maximum (dark arcs),
// relative to the centre, clamped at 0.
__device__ __forceinline__ uint32_t fast_strength2(const uint32_t *c) {
    constexpr int P = kT2Pitch;
    uint32_t p[16];
    p[0] = c[3 * P];       p[1] = c[3 * P + 1];    p[2] = c[2 * P + 2];    p[3] = c[P + 3];
    p[4] = c[3];           p[5] = c[-P + 3];       p[6] = c[-2 * P + 2];   p[7] = c[-3 * P + 1];
    p[8] = c[-3 * P];      p[9] = c[-3 * P - 1];   p[10] = c[-2 * P - 2];  p[11] = c[-P - 3];
    p[12] = c[-3];         p[13] = c[P - 3];       p[14] = c[2 * P - 2];   p[15] = c[3 * P - 1];
    const uint32_t v = c[0];
    // max over the 16 windows of the window minimum, four windows at a time: the windows starting at b..b+3 share
    // the six pixels p[b+3..b+8]; what is left of them are the four 3-windows of (p[b], p[b+1], p[b+2], p[b+9],
    // p[b+10], p[b+11]), and max(min(s0,s1,s2), min(s1,s2,s3)) = min(s1, s2, max(s0,s3)).  8 operations per group,
    // 34 per polarity (the plain two-level sliding minimum needs 40).
    uint32_t glo[4], ghi[4];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        const int b = 4 * g;
        const uint32_t s0 = p[b], s1 = p[b + 1], s2 = p[b + 2], s3 = p[(b + 9) & 15], s4 = p[(b + 10) & 15], s5 = p[(b + 11) & 15];
        const uint32_t q0 = p[b + 3], q1 = p[(b + 4) & 15], q2 = p[(b + 5) & 15], q3 = p[(b + 6) & 15], q4 = p[(b + 7) & 15], q5 = p[(b + 8) & 15];
        glo[g] = min3(max2(min3(max2(s0, s3), s1, s2), min3(max2(s2, s5), s3, s4)), min3(q0, q1, q2), min3(q3, q4, q5));
        ghi[g] = max3(min2(max3(min2(s0, s3), s1, s2), max3(min2(s2, s5), s3, s4)), max3(q0, q1, q2), max3(q3, q4, q5));
    }
    const uint32_t best_lo = max3(glo[0], glo[1], max2(glo[2], glo[3]));
    const uint32_t best_hi = min3(ghi[0], ghi[1], min2(ghi[2], ghi[3]));
    // per lane: max(best_lo - v, v - best_hi, 0); the max/min with v keeps both differences non-negative (no borrow)
    return max2(max2(best_lo, v) - v, v - min2(best_hi, v));
}

// thread -> (row, pair column) of a sweep: row = t / S by a multiply-high with ceil(2^32 / S); S is a multiple of 4
__constant__ uint32_t kRcpS[kMaxS / 4 + 1] = {0u, 0x40000000u, 0x20000000u, 0x15555556u, 0x10000000u, 0x0CCCCCCDu, 0x0AAAAAABu, 0x0924924Au};
__constant__ uint8_t kRowsPerSweep[kMaxS / 4 + 1] = {0, 40, 20, 13, 10, 8, 6, 5};   // kFastThreads / S

// Geometry of one FAST cell from the level tables (kernel parameters): no dependent global load.  Valid cells of a level
// form a rows_eff x cols_eff prefix of the reference's grid (:811-828).
struct CellGeom {
    int level, x0, y0, cw, ch;
};
__device__ __forceinline__ CellGeom cell_geom(const FrameGeom &g, int cell_block) {
    CellGeom c;
    int level = 0;       // cell_begin of the levels past nlevels is INT_MAX (vsg_api.cu)
#pragma unroll
    for (int l = 1; l < 8; ++l) level += cell_block >= g.lv[l].cell_begin ? 1 : 0;
    for (int l = 8; l < g.nlevels; ++l) level += cell_block >= g.lv[l].cell_begin ? 1 : 0;
    const LevelGeom &L = g.lv[level];
    const int local = cell_block - L.cell_begin;
    const int ci = (int)__umulhi((uint32_t)local, L.cols_rcp), cj = local - ci * L.cols_eff;
    c.level = level;
    c.x0 = kBorderMin + cj * L.w_cell;
    c.y0 = kBorderMin + ci * L.h_cell;
    c.cw = min(c.x0 + L.w_cell + 6, L.w - kBorderMin) - c.x0;
    c.ch = min(c.y0 + L.h_cell + 6, L.h - kBorderMin) - c.y0;
    return c;
}

// One FAST cell (kFastThreads threads).
//
// Work layout: thread t owns pair column j = t % S and walks down the cell in sweeps of RB = kFastThreads / S rows
// (rows t / S, t / S + RB, ...), for the strength pass and again for the NMS pass.  The column never changes, so the
// column masks, the shared-memory pointers and the survivor coordinates need no per-iteration index arithmetic: one
// pointer increment per sweep.
//
// The cell window is read straight from global memory: the level's pyramid plane, or the caller's level 0.
__device__ __forceinline__ void fast_cell_body(const FrameGeom &g, const CellGeom &cell, const uint8_t *__restrict__ lvl0_base,
                                               int lvl0_pitch, int64_t lvl0_stride, const uint8_t *__restrict__ pyr,
                                               uint32_t *t2, uint32_t *s2, uint32_t *list, Cand *__restrict__ cand,
                                               int *__restrict__ cand_count, int ini_th, int min_th, int list_cap, int frame) {
    __shared__ int s_count, s_base;
    const int level = cell.level, x0 = cell.x0, y0 = cell.y0, cw = cell.cw, ch = cell.ch;
    const LevelGeom &L = g.lv[level];
    const int tid = threadIdx.x;
    const int iw = cw - 6, ih = ch - 6;            // interior = FAST's [3,w-3) x [3,h-3)
    // lane 0 of a pair holds window column b, lane 1 column b + S; S is a multiple of 4 so that both halves of
    // four consecutive pairs come from two aligned 32-bit loads
    const int S = (((iw + 1) >> 1) + 3) & ~3;
    const int ax0 = x0 & ~3;                       // 4-byte aligned origin of the pair columns
    const int xoff = x0 - ax0;                     // window column w sits at pair column xoff + w
    {
        const int nq = (xoff + S + 6 + 3) >> 2;    // quads of pair columns per row (7..9 typical, <= 12)
        // thread -> (row, quad) by shift/mask: 8 (or 16) quad slots per row, threads beyond nq idle
        const int lq = nq <= 8 ? 3 : 4;
        const int q = tid & ((1 << lq) - 1), r0 = tid >> lq, rstep = kFastThreads >> lq;
        const bool qok = q < nq;
        auto relayout = [&](uint32_t a, uint32_t b, uint32_t *dst) {
            uint4 o;
            o.x = __byte_perm(a, b, 0x7470) & 0x00FF00FFu;   // [a0, -, b0, -]
            o.y = __byte_perm(a, b, 0x7571) & 0x00FF00FFu;
            o.z = __byte_perm(a, b, 0x7672) & 0x00FF00FFu;
            o.w = __byte_perm(a, b, 0x7773) & 0x00FF00FFu;
            *reinterpret_cast<uint4 *>(dst) = o;
        };
        const uint8_t *src;
        int spitch;
        if (level == 0) { src = lvl0_base + (int64_t)frame * lvl0_stride; spitch = lvl0_pitch; }
        else { src = pyr + L.plane_offset + (int64_t)frame * L.plane_stride; spitch = L.pitch; }
        const uint8_t *base = src + (int64_t)y0 * spitch + ax0;
        const uint8_t *row = base + (int64_t)r0 * spitch + 4 * q;
        const int64_t rinc = (int64_t)rstep * spitch;
        uint32_t *dst = t2 + r0 * kT2Pitch + 4 * q;
        // all global loads of the CTA are issued before the first one is consumed
        constexpr int kLoadIters = 3;              // 3 x 20 rows of 8 quads cover the usual 44-row cell without a loop
        uint32_t a[kLoadIters], b[kLoadIters];
#pragma unroll
        for (int it = 0; it < kLoadIters; ++it) {
            if (qok && r0 + it * rstep < ch) {
                a[it] = __ldg(reinterpret_cast<const uint32_t *>(row + it * rinc));
                // the second half may reach past the window, never past the image row (x0 + cw <= W - 16)
                b[it] = __ldg(reinterpret_cast<const uint32_t *>(row + it * rinc + S));
            }
        }
#pragma unroll
        for (int it = 0; it < kLoadIters; ++it)
            if (qok && r0 + it * rstep < ch) relayout(a[it], b[it], dst + it * rstep * kT2Pitch);
        for (int r = r0 + kLoadIters * rstep; qok && r < ch; r += rstep) {   // taller cells
            const uint8_t *rp = base + (int64_t)r * spitch + 4 * q;
            relayout(__ldg(reinterpret_cast<const uint32_t *>(rp)), __ldg(reinterpret_cast<const uint32_t *>(rp + S)),
                     t2 + r * kT2Pitch + 4 * q);
        }
    }
    for (int i = tid; i < kS2Pitch; i += kFastThreads) {     // top and bottom apron rows of the strength plane
        s2[i] = 0;
        s2[(ih + 1) * kS2Pitch + i] = 0;
    }
    if (tid == 0) s_count = 0;

    // this thread's place in a sweep
    const int RB = kRowsPerSweep[S >> 2];
    const int trow = (int)__umulhi((uint32_t)tid, kRcpS[S >> 2]);
    const int j = tid - trow * S;
    const int row0 = trow < RB ? trow : ih;                  // the last kFastThreads - S * RB threads sit the sweeps out
    // lane 0 is interior column j, lane 1 column j + S; columns >= iw do not exist
    const uint32_t kmask = (j < iw ? 0x0000FFFFu : 0u) | (j + S < iw ? 0xFFFF0000u : 0u);
    __syncthreads();

    {
        const uint32_t *c = t2 + (3 + row0) * kT2Pitch + xoff + 3 + j;   // pair (row, interior column j)
        uint32_t *k = s2 + (row0 + 1) * kS2Pitch + j + 1;
        // the two halves meet in the middle: column S-1 (lane 0 of the last pair) and column S (lane 1 of the first pair)
        // are neighbours; their owners also write the two apron pairs of the row
        const bool first = j == 0, last = j == S - 1;
        for (int row = row0; row < ih; row += RB, c += RB * kT2Pitch, k += RB * kS2Pitch) {
            const uint32_t K = fast_strength2(c) & kmask;
            *k = K;
            if (last) k[-S] = K << 16;      // left apron:  lane 0 = outside the cell (0), lane 1 = K(S-1)
            if (first) k[S] = K >> 16;      // right apron: lane 0 = K(S), lane 1 = outside the cell (0)
        }
    }
    __syncthreads();

    for (int pass = 0; pass < 2; ++pass) {
        const int t = pass == 0 ? ini_th : min_th;
        const int tt = max(t, 1);       // a corner scoring 0 (K == 1, only possible at t == 0) never survives the NMS
        // Per sweep the pair's two survivor flags are produced in packed form — K - min(K, max(nb, tt)) is non-zero in
        // a lane iff that pixel beats the threshold and all 8 neighbours — and accumulated as bit `sweep` of the two
        // 16-bit lanes of acc by a multiply-add (FMA pipe, not the ALU pipe the min/max use).  At most 16 sweeps
        // (checked by the launcher).
        const uint32_t tt2 = (uint32_t)tt * 0x00010001u;
        uint32_t acc = 0, pw = 1;
        const uint32_t *c = s2 + (row0 + 1) * kS2Pitch + j + 1;
        for (int row = row0; row < ih; row += RB, c += RB * kS2Pitch, pw <<= 1) {
            const uint32_t K = c[0];
            // strict maximum over the 8 neighbours: neighbours that are not corners at t are below K anyway
            const uint32_t nb = max3(max3(c[-kS2Pitch - 1], c[-kS2Pitch], c[-kS2Pitch + 1]),
                                     max3(c[-1], c[1], c[kS2Pitch - 1]), max3(c[kS2Pitch], c[kS2Pitch + 1], tt2));
            const uint32_t e = K - min2(K, nb);
            acc += min2(e, 0x00010001u) * pw;
        }
        const int cnt = __popc(acc);
        if (cnt) {
            int pos = atomicAdd(&s_count, cnt);
            uint32_t m0 = acc & 0xFFFFu, m1 = acc >> 16;
            const uint32_t *kcol = s2 + (row0 + 1) * kS2Pitch + j + 1;
            while (m0) {
                const int i = __ffs(m0) - 1;
                m0 &= m0 - 1;
                const uint32_t K = kcol[i * RB * kS2Pitch] & 0xFFFFu;
                list[pos++] = (uint32_t)j | ((uint32_t)(row0 + i * RB) << 8) | ((K - 1) << 16);
            }
            while (m1) {
                const int i = __ffs(m1) - 1;
                m1 &= m1 - 1;
                const uint32_t K = kcol[i * RB * kS2Pitch] >> 16;
                list[pos++] = (uint32_t)(j + S) | ((uint32_t)(row0 + i * RB) << 8) | ((K - 1) << 16);
            }
        }
        __syncthreads();
        if (s_count > 0) break;   // uniform: the retry happens only when the cell is empty (:842)
    }
    const int n = min(s_count, list_cap);
    if (n == 0) return;
    const int slot_idx = frame * g.nlevels + level;
    if (tid == 0) s_base = atomicAdd(&cand_count[slot_idx], n);
    __syncthreads();
    Cand *out = cand + L.cand_offset + (int64_t)frame * g.cand_total;
    for (int i = tid; i < n; i += kFastThreads) {
        const int dst = s_base + i;
        if (dst >= L.cand_cap) break;
        const uint32_t e = list[i];
        Cand c;
        c.x = (unsigned short)(x0 + 3 + (e & 0xff));
        c.y = (unsigned short)(y0 + 3 + ((e >> 8) & 0xff));
        c.score = (unsigned short)(e >> 16);
        c.pad = 0;
        out[dst] = c;
    }
}

// shared-memory carve-up of a FAST CTA: pixel pairs, packed strengths, survivor list
struct FastSmem {
    uint32_t *t2, *s2, *list;
};
__device__ __forceinline__ FastSmem fast_smem(uint8_t *base, int tile_rows) {
    FastSmem m;
    m.t2 = reinterpret_cast<uint32_t *>(base);                            // tile_rows x kT2Pitch pixel pairs
    m.s2 = m.t2 + tile_rows * kT2Pitch;                                   // (ih + 2) x kS2Pitch packed strengths
    m.list = m.s2 + (tile_rows - 4) * kS2Pitch;
    return m;
}

__global__ void __launch_bounds__(kFastThreads, VSG_FAST_MINB) fast_kernel(FrameGeom g,
                                                             const uint8_t *__restrict__ lvl0_base, int lvl0_pitch,
                                                             int64_t lvl0_stride, const uint8_t *__restrict__ pyr,
                                                             Cand *__restrict__ cand, int *__restrict__ cand_count,
                                                             int ini_th, int min_th, int tile_rows, int list_cap) {
    extern __shared__ __align__(16) uint8_t smem[];
    pdl_launch_dependents();
    pdl_wait();
    const FastSmem m = fast_smem(smem, tile_rows);
    fast_cell_body(g, cell_geom(g, blockIdx.x), lvl0_base, lvl0_pitch, lvl0_stride, pyr, m.t2, m.s2, m.list, cand,
                   cand_count, ini_th, min_th, list_cap, blockIdx.y);
}

// FAST cells and Gaussian-blur blocks of the same frames in ONE grid.  The two are independent (both only read the
// pyramid) and stress different units — FAST is bound by the ALU pipe (packed min/max), the blur by load latency and
// the FMA pipe (IDP4A / IMAD) — so blur blocks are interleaved between FAST cells, `ratio` cells then one blur block,
// and every SM holds a mix of both.  unit x of a frame -> role:
//   x < nblur * (ratio + 1):  group x / (ratio + 1); position x % (ratio + 1) < ratio is cell group*ratio + position,
//                             position == ratio is blur block `group`;
//   beyond that:              the remaining cells.
struct UnitRole {
    bool blur;
    int index;     // blur block or cell
};
__device__ __forceinline__ UnitRole unit_role(int x, int nblur, int ratio, uint32_t group_rcp) {
    const int group = ratio + 1;
    UnitRole r;
    if (x < nblur * group) {
        const int gi = group == 1 ? x : (int)__umulhi((uint32_t)x, group_rcp), pos = x - gi * group;   // x / group
        r.blur = pos == ratio;
        r.index = r.blur ? gi : gi * ratio + pos;
    } else {
        r.blur = false;
        r.index = nblur * ratio + (x - nblur * group);
    }
    return r;
}

__global__ void __launch_bounds__(kFastThreads, VSG_FAST_MINB) fast_blur_kernel(FrameGeom g, BlurLevels bl,
                                                                  const uint8_t *__restrict__ lvl0_base, int lvl0_pitch,
                                                                  int64_t lvl0_stride, const uint8_t *__restrict__ pyr,
                                                                  uint8_t *__restrict__ blur, Cand *__restrict__ cand,
                                                                  int *__restrict__ cand_count, int ini_th, int min_th,
                                                                  int tile_rows, int list_cap, int nblur, int ratio,
                                                                  uint32_t group_rcp) {
    extern __shared__ __align__(16) uint8_t smem[];
    pdl_launch_dependents();
    pdl_wait();
    const UnitRole role = unit_role(blockIdx.x, nblur, ratio, group_rcp);
    if (role.blur) {
        blur_block_body(g, bl, lvl0_base, lvl0_pitch, lvl0_stride, pyr, blur, role.index, blockIdx.y);
        return;
    }
    const FastSmem m = fast_smem(smem, tile_rows);
    fast_cell_body(g, cell_geom(g, role.index), lvl0_base, lvl0_pitch, lvl0_stride, pyr, m.t2, m.s2, m.list, cand,
                   cand_count, ini_th, min_th, list_cap, blockIdx.y);
}

// blur == nullptr: FAST alone; otherwise the fused FAST + blur grid.
vsg_status launch_fast(const FrameGeom &g, const uint8_t *lvl0_base, int lvl0_pitch, int64_t lvl0_stride, const uint8_t *pyr,
                       uint8_t *blur, Cand *cand, int *cand_count, int ini_th, int min_th, int max_cw, int max_ch, int nframes,
                       cudaStream_t s) {
    if (g.ncells == 0) {
        if (blur) launch_blur(g, lvl0_base, lvl0_pitch, lvl0_stride, pyr, blur, nframes, s);
        return VSG_OK;
    }
    const int max_S = ((((max_cw - 6) + 1) >> 1) + 3) & ~3;
    // at most 16 sweeps of kFastThreads / S rows (the survivor flags of a thread are the 16-bit lanes of one register)
    if (3 + max_S + 6 + 3 > kT2Pitch || max_S + 2 > kS2Pitch || max_S > kMaxS || (max_ch - 6) > 16 * (kFastThreads / max_S)) {
        set_error("FAST cell larger than the shared-memory tile / the 16-sweep survivor masks");
        return VSG_ERR_INVALID;
    }
    const int tile_rows = max_ch;
    const int list_cap = ((max_cw - 6 + 1) / 2) * ((max_ch - 6 + 1) / 2) + 1;
    const size_t smem = (size_t)tile_rows * kT2Pitch * 4 + (size_t)(tile_rows - 4) * kS2Pitch * 4 + (size_t)list_cap * 4 + 16;
    if (smem > 48 * 1024) {   // per device and cheap: set on every launch rather than caching it in a (racy) static
        cudaFuncSetAttribute(fast_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(fast_blur_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    }
    if (!blur) {
        launch_kernel(fast_kernel, dim3(g.ncells, nframes), dim3(kFastThreads), smem, s, true, g, lvl0_base, lvl0_pitch,
                      lvl0_stride, pyr, cand, cand_count, ini_th, min_th, tile_rows, list_cap);
    } else {
        const BlurLevels bl = make_blur_levels(g, nframes, kFastThreads);   // blur blocks of the fused grid have the FAST block size
        const int nblur = bl.block_begin[g.nlevels];
        const int ratio = g.ncells / nblur;
        const uint32_t group_rcp = (uint32_t)((0x100000000ull + (uint64_t)ratio) / (uint64_t)(ratio + 1));   // ceil(2^32 / group)
        launch_kernel(fast_blur_kernel, dim3(g.ncells + nblur, nframes), dim3(kFastThreads), smem, s, true, g, bl, lvl0_base,
                      lvl0_pitch, lvl0_stride, pyr, blur, cand, cand_count, ini_th, min_th, tile_rows, list_cap, nblur, ratio,
                      group_rcp);
    }
    count_launch();
    return VSG_OK;
}

}  // namespace vsg
