// vsg_api.cu — the C ABI of libvsg_cuda.so (include/vsg_cuda.h): extractor object, host-side tables
// and orchestration of the kernels in pyramid.cu / fast.cu / octree.cu / describe.cu.
//
// Reference (snt-arg/visual_sgraphs):
//   ORBextractor::ORBextractor   orb_slam3/src/ORBextractor.cc:411-470   -> build_tables()
//   ORBextractor::operator()     :1083-1169                               -> run_batch()
//   ComputePyramid level sizes   :1171-1180                               -> configure_shape()
//   cell grid                    :795-828                                 -> configure_shape()
//   cv::resize coefficient tables (SURVEY Appendix A1)                    -> build_resize_tables()
// There is no CPU compute path in this library: every entry point that produces results launches
// CUDA kernels and fails with VSG_ERR_CUDA when no device is usable.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "vsg_internal.cuh"

namespace vsg {

static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
bool cuda_ok(cudaError_t e, const char *what) {
    if (e == cudaSuccess) return true;
    set_error("%s: %s", what, cudaGetErrorString(e));
    return false;
}
void count_launch(int n) { g_launches += n; }
// Programmatic dependent launch pays where launch latency is the cost — a handful of frames: 229 -> 213 us per
// single-frame call — and hurts where the kernels are long: with 512 frames per launch the early-resident blocks of the
// next kernel take 10 % off the batch rate (4.24 vs 3.85 ms per batch).  So only batches of up to kPdlMaxFrames frames use it.
static thread_local bool g_pdl_small_batch = true;
constexpr int kPdlMaxFrames = 8;
void pdl_scope(int nframes) { g_pdl_small_batch = nframes <= kPdlMaxFrames; }
bool pdl_enabled() { return g_pdl_small_batch; }

static inline int cv_round(float v) { return (int)lrintf(v); }
static inline int cv_round(double v) { return (int)lrint(v); }
static inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

}  // namespace vsg

using namespace vsg;

struct vsg_extractor {
    int device = 0;
    int max_batch = 1;
    cudaStream_t stream = nullptr;
    // Host-pointer batches are cut into chunks that rotate over `stream` and these two, so that one chunk's H2D,
    // another's kernels and a third's D2H overlap (each chunk works on its own frame range of the scratch buffers).
    static constexpr int kAuxStreams = 2;
    cudaStream_t aux[kAuxStreams] = {nullptr, nullptr};
    int chunk_frames = 128;            // launches of 64 frames reach 76 % of the 512-frame rate, 128: 89 %, 256: 96 %
    uint8_t *color_d = nullptr;        // device staging of colour frames (vsg_extract_batch_color), allocated on first use
    size_t color_bytes = 0;
    // rectification maps (vsg_extractor_set_rectify_map): quantised on the host, resident on the device; independent of the
    // configured shape (the map size IS the shape the rectified frames are extracted at)
    uint32_t *rect_xy[2] = {nullptr, nullptr};
    uint16_t *rect_frac[2] = {nullptr, nullptr};
    int rect_w = 0, rect_h = 0;
    cudaEvent_t fork_ev = nullptr;
    vsg_orb_params p{};
    std::vector<float> scale, inv_scale, sigma2, inv_sigma2;
    std::vector<int> quota;

    // shape dependent state
    int cur_w = 0, cur_h = 0;
    FrameGeom g{};
    int max_cw = 0, max_ch = 0, max_nodes = 0;
    int64_t pyr_bytes_per_frame = 0;

    short4 *tabs_d = nullptr;
    PyrTile *pyr_tiles_d = nullptr;        // one-launch pyramid for small batches (pyramid.cu); nullptr = not available
    int pyr_ntiles = 0, pyr_tile_buf = 0;
    size_t pyr_tile_smem = 0;
    uint8_t *pyr = nullptr, *blur = nullptr;
    Cand *cand = nullptr;
    unsigned short *node_of = nullptr;
    int *cand_count = nullptr;
    LevelKp *level_kps = nullptr;
    int *level_kp_count = nullptr;
    int *slot = nullptr;
    uint8_t *out_block_d = nullptr, *out_block_h = nullptr;   // kps / desc / n / mono below are sub-ranges of these
    size_t out_block_bytes = 0;
    vsg_keypoint *kps_d = nullptr;
    uint8_t *desc_d = nullptr;
    int *n_d = nullptr, *mono_d = nullptr;
    // pinned staging for results
    vsg_keypoint *kps_h = nullptr;
    uint8_t *desc_h = nullptr;
    int *n_h = nullptr, *mono_h = nullptr;

    // optional per-stage timing: a ring of event sets, harvested lazily
    bool profile = false;
    static constexpr int kEvRing = 32;
    cudaEvent_t ev[kEvRing][VSG_NUM_STAGES + 1] = {};
    bool ev_created = false;
    int ev_head = 0, ev_pending = 0;
    double stage_ms[VSG_NUM_STAGES] = {0, 0, 0, 0, 0};
    int64_t stage_runs = 0;

    void harvest_one() {   // oldest pending event set -> accumulators (blocks until it completed)
        const int slot = (ev_head - ev_pending + 2 * kEvRing) % kEvRing;
        cudaEventSynchronize(ev[slot][VSG_NUM_STAGES]);
        for (int k = 0; k < VSG_NUM_STAGES; ++k) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, ev[slot][k], ev[slot][k + 1]);
            stage_ms[k] += ms;
        }
        ++stage_runs;
        --ev_pending;
    }

    // where level 0 of the last call lives
    const uint8_t *lvl0_base = nullptr;
    int lvl0_pitch = 0;
    int64_t lvl0_stride = 0;
    int last_nframes = 0;
    bool results_on_handle = false;    // kps_d / desc_d / n_d hold the last call's results (host-pointer API)

    void free_shape() {
        cudaFree(tabs_d); cudaFree(pyr_tiles_d); cudaFree(pyr); cudaFree(blur); cudaFree(cand); cudaFree(node_of);
        cudaFree(cand_count); cudaFree(level_kps); cudaFree(level_kp_count); cudaFree(slot); cudaFree(out_block_d);
        cudaFree(color_d);
        color_d = nullptr; color_bytes = 0;
        cudaFreeHost(out_block_h);
        out_block_d = out_block_h = nullptr; out_block_bytes = 0;
        tabs_d = nullptr; pyr_tiles_d = nullptr; pyr_ntiles = 0; pyr = blur = nullptr; cand = nullptr; node_of = nullptr;
        cand_count = nullptr; level_kps = nullptr; level_kp_count = nullptr; slot = nullptr; kps_d = nullptr;
        desc_d = nullptr; n_d = mono_d = nullptr; kps_h = nullptr; desc_h = nullptr; n_h = mono_h = nullptr;
        cur_w = cur_h = 0;
    }
};

namespace {

// ORBextractor::ORBextractor — ORBextractor.cc:411-446 (scale tables and per-level quotas)
void build_tables(vsg_extractor *ex) {
    const int nl = ex->p.nlevels;
    const double scale_factor = ex->p.scale_factor;  // the member is a double (ORBextractor.h:105)
    ex->scale.assign(nl, 1.f);
    ex->sigma2.assign(nl, 1.f);
    for (int i = 1; i < nl; ++i) {
        ex->scale[i] = (float)(ex->scale[i - 1] * scale_factor);
        ex->sigma2[i] = ex->scale[i] * ex->scale[i];
    }
    ex->inv_scale.resize(nl);
    ex->inv_sigma2.resize(nl);
    for (int i = 0; i < nl; ++i) {
        ex->inv_scale[i] = 1.0f / ex->scale[i];
        ex->inv_sigma2[i] = 1.0f / ex->sigma2[i];
    }
    ex->quota.assign(nl, 0);
    const float factor = (float)(1.0f / scale_factor);
    float desired = ex->p.nfeatures * (1 - factor) / (1 - (float)std::pow((double)factor, (double)nl));
    int sum = 0;
    for (int l = 0; l < nl - 1; ++l) {
        ex->quota[l] = cv_round(desired);
        sum += ex->quota[l];
        desired *= factor;
    }
    ex->quota[nl - 1] = std::max(ex->p.nfeatures - sum, 0);
}

// cv::resize INTER_LINEAR coefficient tables — SURVEY Appendix A1
void build_resize_tables(int sw, int sh, int dw, int dh, int dw_pad, std::vector<short4> &xt, std::vector<short4> &yt) {
    const double scale_x = 1.0 / ((double)dw / sw), scale_y = 1.0 / ((double)dh / sh);
    xt.resize(dw_pad);
    yt.resize(dh);
    for (int dx = 0; dx < dw_pad; ++dx) {
        const int x = std::min(dx, dw - 1);  // pad entries repeat the last column (results land in pitch padding)
        float fx = (float)((x + 0.5) * scale_x - 0.5);
        int sx = (int)std::floor(fx);
        fx -= sx;
        if (sx < 0) { fx = 0; sx = 0; }
        if (sx >= sw - 1) { fx = 0; sx = sw - 1; }
        xt[dx] = make_short4((short)sx, (short)std::min(sx + 1, sw - 1), (short)cv_round((1.f - fx) * 2048.f),
                             (short)cv_round(fx * 2048.f));
    }
    for (int dy = 0; dy < dh; ++dy) {
        float fy = (float)((dy + 0.5) * scale_y - 0.5);
        int sy = (int)std::floor(fy);
        fy -= sy;
        const int sy0 = std::min(std::max(sy, 0), sh - 1), sy1 = std::min(std::max(sy + 1, 0), sh - 1);
        yt[dy] = make_short4((short)sy0, (short)sy1, (short)cv_round((1.f - fy) * 2048.f), (short)cv_round(fy * 2048.f));
    }
}

vsg_status configure_shape(vsg_extractor *ex, int w, int h) {
    if (ex->cur_w == w && ex->cur_h == h) return VSG_OK;
    if (w > kMaxImageDim || h > kMaxImageDim) {   // candidate / node coordinates and the resize tables are 16-bit (15 in the oct-tree)
        set_error("image %dx%d too large: at most %d pixels per side", w, h, kMaxImageDim);
        return VSG_ERR_INVALID;
    }
    CK(cudaSetDevice(ex->device));
    int smem_optin = 0;
    size_t octree_static = 0;
    CK(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, ex->device));
    const vsg_status ost = octree_static_smem_bytes(&octree_static);
    if (ost != VSG_OK) return ost;
    ex->free_shape();
    const int nl = ex->p.nlevels;
    FrameGeom &g = ex->g;
    memset(&g, 0, sizeof(g));
    g.nlevels = nl;
    std::vector<Cell> cells;
    ex->max_cw = ex->max_ch = 7;
    ex->max_nodes = 8;
    int64_t plane_off = 0, cand_off = 0;
    int kp_off = 0;
    std::vector<std::vector<short4>> xts(nl), yts(nl);
    for (int l = 0; l < nl; ++l) {
        LevelGeom &L = g.lv[l];
        L.w = cv_round((float)w * ex->inv_scale[l]);   // :1176
        L.h = cv_round((float)h * ex->inv_scale[l]);
        const int min_b = kBorderMin, max_bx = L.w - kBorderMin, max_by = L.h - kBorderMin;
        const float width = (float)(max_bx - min_b), height = (float)(max_by - min_b);
        if (width < 35.f || height < 35.f) {
            set_error("image %dx%d too small: level %d is %dx%d (needs >= 67x67 for one 35-px cell)", w, h, l, L.w, L.h);
            return VSG_ERR_INVALID;
        }
        L.pitch = (int)align_up(L.w, 64);
        L.plane_stride = align_up((int64_t)L.pitch * L.h, 256);
        L.plane_offset = plane_off;
        plane_off += L.plane_stride * ex->max_batch;
        L.n_cols = (int)(width / 35.f);                // :803-809
        L.n_rows = (int)(height / 35.f);
        L.w_cell = (int)std::ceil(width / L.n_cols);
        L.h_cell = (int)std::ceil(height / L.n_rows);
        L.cell_begin = (int)cells.size();
        int cand_cap = 0;
        for (int i = 0; i < L.n_rows; ++i) {           // :811-828
            const float ini_y = (float)(min_b + i * L.h_cell);
            float max_y = ini_y + L.h_cell + 6;
            if (ini_y >= max_by - 3) continue;
            if (max_y > max_by) max_y = (float)max_by;
            for (int j = 0; j < L.n_cols; ++j) {
                const float ini_x = (float)(min_b + j * L.w_cell);
                float max_x = ini_x + L.w_cell + 6;
                if (ini_x >= max_bx - 6) continue;
                if (max_x > max_bx) max_x = (float)max_bx;
                Cell c;
                c.level = (short)l;
                c.x0 = (short)ini_x; c.y0 = (short)ini_y;
                c.cw = (short)((int)max_x - (int)ini_x); c.ch = (short)((int)max_y - (int)ini_y);
                c.pad = 0;
                if (c.cw < 7 || c.ch < 7) continue;   // cv::FAST finds nothing in such a window
                cells.push_back(c);
                ex->max_cw = std::max<int>(ex->max_cw, c.cw);
                ex->max_ch = std::max<int>(ex->max_ch, c.ch);
                cand_cap += ((c.cw - 6 + 1) / 2) * ((c.ch - 6 + 1) / 2);
            }
        }
        L.cell_count = (int)cells.size() - L.cell_begin;
        L.cols_eff = L.rows_eff = 0;
        for (int k = L.cell_begin; k < (int)cells.size(); ++k) {
            const Cell &c = cells[k];
            L.cols_eff = std::max(L.cols_eff, (c.x0 - min_b) / L.w_cell + 1);
            L.rows_eff = std::max(L.rows_eff, (c.y0 - min_b) / L.h_cell + 1);
        }
        if (L.cols_eff * L.rows_eff != L.cell_count) {
            set_error("internal: level %d cell table is not a prefix rectangle", l);
            return VSG_ERR_INVALID;
        }
        L.cols_rcp = (uint32_t)((0x100000000ull + (uint64_t)L.cols_eff - 1) / (uint64_t)std::max(L.cols_eff, 1));
        L.wcell_rcp = L.w_cell > 1 ? (uint32_t)((0x100000000ull + (uint64_t)L.w_cell - 1) / (uint64_t)L.w_cell) : 0xFFFFFFFFu;
        L.hcell_rcp = L.h_cell > 1 ? (uint32_t)((0x100000000ull + (uint64_t)L.h_cell - 1) / (uint64_t)L.h_cell) : 0xFFFFFFFFu;
        L.quota = ex->quota[l];
        L.n_ini = (int)std::round(static_cast<float>(max_bx - min_b) / (max_by - min_b));   // :566
        if (L.n_ini < 1) {
            set_error("image %dx%d: aspect ratio below 0.5 is not supported by the reference oct-tree (nIni = 0)", w, h);
            return VSG_ERR_INVALID;
        }
        L.h_x = static_cast<float>(max_bx - min_b) / L.n_ini;                                // :568
        L.cand_cap = cand_cap + 8;
        L.cand_offset = cand_off;
        cand_off += L.cand_cap;
        L.kp_cap = std::max(L.quota, 4 * L.n_ini) + 4;
        L.kp_offset = kp_off;
        kp_off += L.kp_cap;
        // the oct-tree keeps a level's nodes in shared memory; a quota whose lists do not fit cannot be launched
        const size_t octree_need = octree_smem_bytes(L.kp_cap + 4) + octree_static;
        if (octree_need > (size_t)smem_optin) {
            set_error("level %d: oct-tree quota %d needs %zu bytes of shared memory per block, the device allows %d", l, L.quota,
                      octree_need, smem_optin);
            return VSG_ERR_INVALID;
        }
        ex->max_nodes = std::max(ex->max_nodes, L.kp_cap + 4);
        L.scale = ex->scale[l];
        L.kp_size = (float)(int)(kPatch * ex->scale[l]);                                    // :884
        L.resize_tma_ok = 0;
        if (l > 0) {
            build_resize_tables(g.lv[l - 1].w, g.lv[l - 1].h, L.w, L.h, (int)align_up(L.w, 4), xts[l], yts[l]);
            L.resize_tma_ok = resize_tma_fits(xts[l], yts[l], L.w, L.h) ? 1 : 0;
        }
    }
    g.ncells = (int)cells.size();
    for (int l = nl; l < kMaxLevels; ++l) g.lv[l].cell_begin = 0x7fffffff;   // fast.cu finds a cell's level by counting begins <= cell
    g.cand_total = cand_off;
    g.kp_total = kp_off;
    g.out_cap = kp_off;
    ex->pyr_bytes_per_frame = plane_off / ex->max_batch;

    const int B = ex->max_batch;
    // resize tables, one allocation
    size_t ntab = 0;
    for (int l = 1; l < nl; ++l) ntab += xts[l].size() + yts[l].size();
    CK(cudaMalloc(&ex->tabs_d, std::max<size_t>(ntab, 1) * sizeof(short4)));
    size_t toff = 0;
    for (int l = 1; l < nl; ++l) {
        CK(cudaMemcpy(ex->tabs_d + toff, xts[l].data(), xts[l].size() * sizeof(short4), cudaMemcpyHostToDevice));
        g.lv[l].xtab = ex->tabs_d + toff;
        toff += xts[l].size();
        CK(cudaMemcpy(ex->tabs_d + toff, yts[l].data(), yts[l].size() * sizeof(short4), cudaMemcpyHostToDevice));
        g.lv[l].ytab = ex->tabs_d + toff;
        toff += yts[l].size();
    }
    // tiles of the one-launch pyramid: a 12 x 12 partition of every level; going down from the top level, a tile's region
    // is the bounding box of what it owns and of the taps of its region one level up
    if (nl >= 2) {
        constexpr int ntx = 12, nty = 12;
        std::vector<PyrTile> tiles((size_t)ntx * nty);
        int buf = 0, ntab_max = 0, dim_max = 0;
        for (int ty = 0; ty < nty; ++ty)
            for (int tx = 0; tx < ntx; ++tx) {
                PyrTile &t = tiles[(size_t)ty * ntx + tx];
                int ntab_t = 0;
                for (int l = nl - 1; l >= 0; --l) {
                    const int W = g.lv[l].w, H = g.lv[l].h;
                    PyrTileBox o{(short)(tx * W / ntx), (short)(ty * H / nty), (short)((tx + 1) * W / ntx - 1), (short)((ty + 1) * H / nty - 1)};
                    PyrTileBox r = o;
                    if (l < nl - 1) {
                        const PyrTileBox &u = t.region[l + 1];
                        const short nx0 = xts[l + 1][u.x0].x, nx1 = xts[l + 1][u.x1].y, ny0 = yts[l + 1][u.y0].x, ny1 = yts[l + 1][u.y1].y;
                        if (l == 0) r = PyrTileBox{nx0, ny0, nx1, ny1};      // nothing is stored at level 0
                        else r = PyrTileBox{std::min(o.x0, nx0), std::min(o.y0, ny0), std::max(o.x1, nx1), std::max(o.y1, ny1)};
                    }
                    t.owned[l] = o;
                    t.region[l] = r;
                    t.rcp_w[l] = (uint32_t)((0x100000000ull + (uint64_t)(r.x1 - r.x0)) / (uint64_t)(r.x1 - r.x0 + 1));
                    buf = std::max(buf, (r.x1 - r.x0 + 1) * (r.y1 - r.y0 + 1));
                    if (l > 0) dim_max = std::max(dim_max, std::max(r.x1 - r.x0 + 1, r.y1 - r.y0 + 1));
                    if (l > 0) ntab_t += (r.x1 - r.x0 + 1) + (r.y1 - r.y0 + 1);
                }
                for (int l = nl; l < kMaxLevels; ++l) { t.owned[l] = t.region[l] = PyrTileBox{0, 0, -1, -1}; t.rcp_w[l] = 0; }
                ntab_max = std::max(ntab_max, ntab_t);
            }
        ex->pyr_tile_buf = (int)align_up(buf, 16);
        ex->pyr_tile_smem = 2 * (size_t)ex->pyr_tile_buf + (size_t)ntab_max * sizeof(short4);
        if (ex->pyr_tile_smem <= 160 * 1024 && dim_max <= 256 && buf < 65536 && nl <= kMaxLevels && g.lv[nl - 1].w >= 2 * ntx && g.lv[nl - 1].h >= 2 * nty) {
            CK(cudaMalloc(&ex->pyr_tiles_d, tiles.size() * sizeof(PyrTile)));
            CK(cudaMemcpy(ex->pyr_tiles_d, tiles.data(), tiles.size() * sizeof(PyrTile), cudaMemcpyHostToDevice));
            ex->pyr_ntiles = (int)tiles.size();
        }
    }
    CK(cudaMalloc(&ex->pyr, plane_off + 256));
    CK(cudaMalloc(&ex->blur, plane_off + 256));
    CK(cudaMemset(ex->pyr, 0, plane_off + 256));
    CK(cudaMalloc(&ex->cand, (size_t)g.cand_total * B * sizeof(Cand)));
    CK(cudaMalloc(&ex->node_of, (size_t)g.cand_total * B * sizeof(unsigned short)));
    CK(cudaMalloc(&ex->cand_count, (size_t)B * nl * sizeof(int)));
    CK(cudaMalloc(&ex->level_kps, (size_t)g.kp_total * B * sizeof(LevelKp)));
    CK(cudaMalloc(&ex->level_kp_count, (size_t)B * nl * sizeof(int)));
    CK(cudaMalloc(&ex->slot, (size_t)g.kp_total * B * sizeof(int)));
    // The four result arrays are sub-ranges of ONE device block and of ONE pinned host block with the same layout, so a
    // call that fills the whole handle (a single frame on a max_batch = 1 handle, above all) brings everything back with
    // a single device-to-host copy instead of four.
    {
        auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
        const size_t off_desc = up((size_t)g.out_cap * B * sizeof(vsg_keypoint));
        const size_t off_n = off_desc + up((size_t)g.out_cap * B * 32);
        const size_t off_mono = off_n + up((size_t)B * sizeof(int));
        ex->out_block_bytes = off_mono + up((size_t)B * sizeof(int));
        CK(cudaMalloc(&ex->out_block_d, ex->out_block_bytes));
        CK(cudaMallocHost(&ex->out_block_h, ex->out_block_bytes));
        ex->kps_d = reinterpret_cast<vsg_keypoint *>(ex->out_block_d);
        ex->desc_d = ex->out_block_d + off_desc;
        ex->n_d = reinterpret_cast<int *>(ex->out_block_d + off_n);
        ex->mono_d = reinterpret_cast<int *>(ex->out_block_d + off_mono);
        ex->kps_h = reinterpret_cast<vsg_keypoint *>(ex->out_block_h);
        ex->desc_h = ex->out_block_h + off_desc;
        ex->n_h = reinterpret_cast<int *>(ex->out_block_h + off_n);
        ex->mono_h = reinterpret_cast<int *>(ex->out_block_h + off_mono);
    }
    ex->cur_w = w;
    ex->cur_h = h;
    return VSG_OK;
}

// The device pipeline for frames [f0, f0 + nframes) of the handle's scratch buffers, on stream `s`.  Level 0 of frame
// f0 is at lvl0_base; the output pointers address frame f0 as well.  Chunks of one batch run this concurrently on
// different streams: every per-frame array is addressed through a geometry whose offsets are shifted to frame f0.
// VSG_PYR_TILE = n: batches of at most n frames build the pyramid in one launch (default 4; 0 = always level by level)
static int pyr_tile_max_frames() {
    const char *e = getenv("VSG_PYR_TILE");
    return e ? atoi(e) : 4;
}

vsg_status run_pipeline(vsg_extractor *ex, cudaStream_t s, int f0, const uint8_t *lvl0_base, int lvl0_pitch,
                        int64_t lvl0_stride, int nframes, int lap_x0, int lap_x1, vsg_keypoint *kps_dev,
                        uint8_t *desc_dev, int out_cap, int *n_dev, int *mono_dev) {
    FrameGeom g = ex->g;
    for (int l = 0; l < g.nlevels; ++l) {
        g.lv[l].plane_offset += (int64_t)f0 * g.lv[l].plane_stride;
        g.lv[l].cand_offset += (int64_t)f0 * g.cand_total;
    }
    pdl_scope(nframes);
    int *cand_count = ex->cand_count + (size_t)f0 * g.nlevels;
    int *level_kp_count = ex->level_kp_count + (size_t)f0 * g.nlevels;
    LevelKp *level_kps = ex->level_kps + (size_t)f0 * g.kp_total;
    int *slot = ex->slot + (size_t)f0 * g.kp_total;
    CK(cudaMemsetAsync(cand_count, 0, (size_t)nframes * g.nlevels * sizeof(int), s));
    cudaEvent_t *ev = nullptr;
    if (ex->profile && s == ex->stream) {
        if (!ex->ev_created) {
            for (int i = 0; i < vsg_extractor::kEvRing; ++i)
                for (int k = 0; k <= VSG_NUM_STAGES; ++k) CK(cudaEventCreate(&ex->ev[i][k]));
            ex->ev_created = true;
        }
        if (ex->ev_pending == vsg_extractor::kEvRing) ex->harvest_one();
        ev = ex->ev[ex->ev_head];
        ex->ev_head = (ex->ev_head + 1) % vsg_extractor::kEvRing;
        ++ex->ev_pending;
    }
#define STAGE_MARK(k) do { if (ev) CK(cudaEventRecord(ev[k], s)); } while (0)
    STAGE_MARK(0);
    if (ex->pyr_tiles_d && nframes <= pyr_tile_max_frames()) {    // ComputePyramid (:1171-1195) in one launch
        launch_pyramid_tiles(g, ex->pyr_tiles_d, ex->pyr_ntiles, ex->pyr_tile_buf, ex->pyr_tile_smem, lvl0_base, lvl0_pitch, lvl0_stride,
                             ex->pyr, nframes, s);
    } else {
        for (int l = 1; l < g.nlevels; ++l) {                     // ... or level by level
            const LevelGeom &P = g.lv[l - 1];
            if (l == 1) launch_resize_level(g, l, lvl0_base, lvl0_pitch, lvl0_stride, ex->pyr, nframes, s);
            else launch_resize_level(g, l, ex->pyr + P.plane_offset, P.pitch, P.plane_stride, ex->pyr, nframes, s);
        }
    }
    STAGE_MARK(1);
    // FAST cells and the Gaussian blur share one grid (fast.cu); large batches blur on the tensor cores instead
    // (blur_tc.cu), as a stage of its own after the oct-tree
    const BlurTcPlan *blur_tc = plan_blur_tc(g, lvl0_base, lvl0_pitch, lvl0_stride, ex->pyr, ex->blur, nframes);
    const vsg_status fst = launch_fast(g, lvl0_base, lvl0_pitch, lvl0_stride, ex->pyr, blur_tc ? nullptr : ex->blur, ex->cand,
                                       cand_count, ex->p.ini_th_fast, ex->p.min_th_fast, ex->max_cw, ex->max_ch, nframes, s);
    if (fst != VSG_OK) return fst;
    STAGE_MARK(2);
    // nothing after this may run when the oct-tree did not: describe reads the level keypoint counts it writes
    const vsg_status ost = launch_octree(g, ex->cand, cand_count, ex->node_of, level_kps, level_kp_count, ex->max_nodes, nframes, s);
    if (ost != VSG_OK) return ost;
    STAGE_MARK(3);
    if (blur_tc) launch_blur_tc(blur_tc, ex->blur, s);
    STAGE_MARK(4);
    launch_describe(g, lvl0_base, lvl0_pitch, lvl0_stride, ex->pyr, ex->blur, level_kps, level_kp_count, lap_x0,
                    lap_x1, kps_dev, desc_dev, out_cap, n_dev, mono_dev, slot, nframes, s);
    STAGE_MARK(5);
#undef STAGE_MARK
    CK(cudaGetLastError());
    return VSG_OK;
}

}  // namespace

namespace vsg {
bool extractor_pyramid(vsg_extractor *ex, PyramidRef *out) {
    if (!ex || ex->cur_w == 0 || ex->last_nframes == 0) return false;
    out->device = ex->device;
    out->nframes = ex->last_nframes;
    out->geom = &ex->g;
    out->lvl0_base = ex->lvl0_base;
    out->lvl0_pitch = ex->lvl0_pitch;
    out->lvl0_stride = ex->lvl0_stride;
    out->pyr = ex->pyr;
    out->scale = ex->scale.data();
    out->inv_scale = ex->inv_scale.data();
    out->stream = ex->stream;
    out->kps_dev = ex->results_on_handle ? ex->kps_d : nullptr;
    out->desc_dev = ex->results_on_handle ? ex->desc_d : nullptr;
    out->n_dev = ex->results_on_handle ? ex->n_d : nullptr;
    out->out_cap = ex->g.out_cap;
    return true;
}
}  // namespace vsg

extern "C" {

const char *vsg_last_error(void) { return g_err; }

int vsg_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int64_t vsg_launch_count(void) { return g_launches.load(); }

vsg_status vsg_extractor_create(const vsg_orb_params *params, int device, int max_batch, vsg_extractor **out) {
    if (!params || !out || max_batch < 1 || params->nlevels < 1 || params->nlevels > kMaxLevels ||
        params->scale_factor <= 1.0f || params->scale_factor >= 2.0f || params->nfeatures < 0) {
        // scale factors >= 2 take cv::resize's INTER_AREA shortcut in the reference and are not restated here
        set_error("vsg_extractor_create: invalid argument");
        return VSG_ERR_INVALID;
    }
    if (vsg_device_count() <= device || device < 0) {
        set_error("vsg_extractor_create: CUDA device %d not available (this library has no CPU fallback)", device);
        return VSG_ERR_CUDA;
    }
    vsg_extractor *ex = new vsg_extractor();
    ex->device = device;
    ex->max_batch = max_batch;
    ex->p = *params;
    build_tables(ex);
    if (!cuda_ok(cudaSetDevice(device), "cudaSetDevice") ||
        !cuda_ok(cudaStreamCreateWithFlags(&ex->stream, cudaStreamNonBlocking), "cudaStreamCreate") ||
        !cuda_ok(cudaStreamCreateWithFlags(&ex->aux[0], cudaStreamNonBlocking), "cudaStreamCreate") ||
        !cuda_ok(cudaStreamCreateWithFlags(&ex->aux[1], cudaStreamNonBlocking), "cudaStreamCreate")) {
        delete ex;
        return VSG_ERR_CUDA;
    }
    if (const char *e = getenv("VSG_CHUNK_FRAMES")) ex->chunk_frames = std::max(1, atoi(e));
    cudaEventCreateWithFlags(&ex->fork_ev, cudaEventDisableTiming);
    *out = ex;
    return VSG_OK;
}

void vsg_extractor_destroy(vsg_extractor *ex) {
    if (!ex) return;
    cudaSetDevice(ex->device);
    if (ex->stream) { cudaStreamSynchronize(ex->stream); cudaStreamDestroy(ex->stream); }
    for (cudaStream_t a : ex->aux)
        if (a) { cudaStreamSynchronize(a); cudaStreamDestroy(a); }
    if (ex->fork_ev) cudaEventDestroy(ex->fork_ev);
    if (ex->ev_created)
        for (int i = 0; i < vsg_extractor::kEvRing; ++i)
            for (int k = 0; k <= VSG_NUM_STAGES; ++k) cudaEventDestroy(ex->ev[i][k]);
    ex->free_shape();
    for (int k = 0; k < 2; ++k) { cudaFree(ex->rect_xy[k]); cudaFree(ex->rect_frac[k]); }
    delete ex;
}

vsg_status vsg_extractor_tables(const vsg_extractor *ex, float *scale, float *inv_scale, float *sigma2,
                                float *inv_sigma2, int32_t *features_per_level) {
    if (!ex) return VSG_ERR_INVALID;
    for (int i = 0; i < ex->p.nlevels; ++i) {
        if (scale) scale[i] = ex->scale[i];
        if (inv_scale) inv_scale[i] = ex->inv_scale[i];
        if (sigma2) sigma2[i] = ex->sigma2[i];
        if (inv_sigma2) inv_sigma2[i] = ex->inv_sigma2[i];
        if (features_per_level) features_per_level[i] = ex->quota[i];
    }
    return VSG_OK;
}

int vsg_extractor_max_keypoints(vsg_extractor *ex, int width, int height) {
    if (!ex) return VSG_ERR_INVALID;
    vsg_status st = configure_shape(ex, width, height);
    if (st != VSG_OK) return st;
    return ex->g.out_cap;
}

// channels == 1: 8-bit gray frames; 3 / 4: interleaved colour frames converted on the device (r_first: the first channel
// is red, i.e. COLOR_RGB2GRAY / COLOR_RGBA2GRAY, else the BGR variants)
// How the frames of a host-pointer batch reach the level-0 planes: copied as they are (gray), through cvtColor (3 / 4
// channels) or through cv::remap with the handle's rectification maps (rect_slots = 1 or 2 cameras; gray input of
// src_w x src_h pixels, the extraction runs at the maps' size).
static vsg_status extract_batch_host(vsg_extractor *ex, const uint8_t *images, int nframes, int src_w, int src_h, int pitch,
                                     size_t frame_stride, int channels, int r_first, int rect_slots, int lap_x0, int lap_x1,
                                     vsg_keypoint *keypoints_out, uint8_t *descriptors_out, int capacity, int *n_out,
                                     int *mono_index_out) {
    if (!ex) return VSG_ERR_INVALID;
    if (!images || src_w <= 0 || src_h <= 0 || nframes <= 0) return VSG_EMPTY_IMAGE;   // :1087-1088
    if (nframes > ex->max_batch || pitch < src_w * channels || capacity < 0 || (channels != 1 && channels != 3 && channels != 4)) {
        set_error("vsg_extract_batch: nframes %d > max_batch %d, or bad pitch/capacity/channels", nframes, ex->max_batch);
        return VSG_ERR_INVALID;
    }
    const bool staged = channels != 1 || rect_slots > 0;               // frames land in the staging buffer first
    const int width = rect_slots > 0 ? ex->rect_w : src_w, height = rect_slots > 0 ? ex->rect_h : src_h;
    CK(cudaSetDevice(ex->device));
    vsg_status st = configure_shape(ex, width, height);
    if (st != VSG_OK) return st;
    const int cpitch = (src_w * channels + 63) & ~63;                   // staging pitch of a colour / unrectified row
    const size_t cstride = (size_t)cpitch * src_h;
    if (staged && ex->color_bytes < cstride * ex->max_batch) {
        cudaFree(ex->color_d);
        ex->color_d = nullptr; ex->color_bytes = 0;
        CK(cudaMalloc(&ex->color_d, cstride * ex->max_batch));
        ex->color_bytes = cstride * ex->max_batch;
    }
    const FrameGeom &g = ex->g;
    const LevelGeom &L0 = g.lv[0];
    uint8_t *lvl0 = ex->pyr + L0.plane_offset;
    ex->lvl0_base = lvl0; ex->lvl0_pitch = L0.pitch; ex->lvl0_stride = L0.plane_stride; ex->last_nframes = nframes;
    ex->results_on_handle = true;
    // Results go straight into the caller's arrays when those are page-locked (one strided D2H each, no
    // host-side copy); otherwise through the handle's pinned staging buffers.
    auto pinned = [](const void *p) {
        if (!p) return false;
        cudaPointerAttributes a;
        if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
        return a.type == cudaMemoryTypeHost;
    };
    const bool direct = capacity >= g.out_cap && (!keypoints_out || pinned(keypoints_out)) &&
                        (!descriptors_out || pinned(descriptors_out));
    // Chunked software pipeline: chunk c runs H2D -> kernels -> D2H on stream c mod 3, on its own frame range.
    // Batches of 128 frames and more are cut into at least two chunks of at most chunk_frames frames (128 frames -> 2 x 64,
    // 256 -> 2 x 128, 512 -> 4 x 128): long enough launches to be efficient, short enough to overlap the copies.
    const int min_chunk = std::min(ex->chunk_frames, 64);
    const bool chunked = !ex->profile && nframes >= 2 * min_chunk;
    int chunk = nframes;
    if (chunked) {
        const int nchunks = std::max(2, (nframes + ex->chunk_frames - 1) / ex->chunk_frames);
        chunk = (nframes + nchunks - 1) / nchunks;
    }
    const bool tight = frame_stride == (size_t)pitch * height && (int64_t)L0.pitch * L0.h == L0.plane_stride;
    RectifyMaps maps = {{ex->rect_xy[0], ex->rect_xy[1]}, {ex->rect_frac[0], ex->rect_frac[1]}, rect_slots};
    int nstreams_used = 0;
    if (chunked) {   // chunks on the aux streams must not start before work already queued on ex->stream (an asynchronous
                     // vsg_extract_batch_dev call) has finished with the shared per-frame scratch
        CK(cudaEventRecord(ex->fork_ev, ex->stream));
        for (cudaStream_t a : ex->aux) CK(cudaStreamWaitEvent(a, ex->fork_ev, 0));
    }
    for (int f0 = 0, c = 0; f0 < nframes; f0 += chunk, ++c) {
        const int nf = std::min(chunk, nframes - f0);
        cudaStream_t s = (c % 3 == 0) ? ex->stream : ex->aux[c % 3 - 1];
        nstreams_used = std::min(3, c + 1);
        uint8_t *dst0 = lvl0 + (int64_t)f0 * L0.plane_stride;
        const uint8_t *src0 = images + (size_t)f0 * frame_stride;
        if (staged) {
            uint8_t *c0 = ex->color_d + (size_t)f0 * cstride;
            if (frame_stride == (size_t)pitch * src_h && pitch == cpitch && pitch == src_w * channels) {
                CK(cudaMemcpyAsync(c0, src0, (size_t)pitch * src_h * nf, cudaMemcpyHostToDevice, s));   // linear, see below
            } else if (frame_stride == (size_t)pitch * src_h) {
                CK(cudaMemcpy2DAsync(c0, cpitch, src0, pitch, (size_t)src_w * channels, (size_t)src_h * nf,
                                     cudaMemcpyHostToDevice, s));
            } else {
                for (int f = 0; f < nf; ++f)
                    CK(cudaMemcpy2DAsync(c0 + f * cstride, cpitch, src0 + f * frame_stride, pitch, (size_t)src_w * channels,
                                         src_h, cudaMemcpyHostToDevice, s));
            }
            if (rect_slots > 0)
                launch_remap(c0, cpitch, (int64_t)cstride, src_w, src_h, maps, f0, dst0, L0.pitch, L0.plane_stride, width, height, nf, s);
            else
                launch_cvt_gray(c0, cpitch, (int64_t)cstride, channels, r_first, dst0, L0.pitch, L0.plane_stride, width, height, nf, s);
        } else if (tight && pitch == width && L0.pitch == width) {
            // one linear copy: a 2-D copy of 640-byte rows runs at two thirds of the PCIe rate of a linear one (36 vs
            // 55 GB/s measured), which used to cap the end-to-end rate below the kernels' rate
            CK(cudaMemcpyAsync(dst0, src0, (size_t)width * height * nf, cudaMemcpyHostToDevice, s));
        } else if (tight) {
            CK(cudaMemcpy2DAsync(dst0, L0.pitch, src0, pitch, width, (size_t)height * nf, cudaMemcpyHostToDevice, s));
        } else {
            for (int f = 0; f < nf; ++f)
                CK(cudaMemcpy2DAsync(dst0 + f * L0.plane_stride, L0.pitch, src0 + f * frame_stride, pitch, width, height,
                                     cudaMemcpyHostToDevice, s));
        }
        vsg_keypoint *kd = ex->kps_d + (size_t)f0 * g.out_cap;
        uint8_t *dd = ex->desc_d + (size_t)f0 * g.out_cap * 32;
        st = run_pipeline(ex, s, f0, dst0, L0.pitch, L0.plane_stride, nf, lap_x0, lap_x1, kd, dd, g.out_cap, ex->n_d + f0,
                          ex->mono_d + f0);
        if (st != VSG_OK) return st;
        if (!direct && nf == ex->max_batch) {     // the call fills the handle: one copy of the whole result block
            CK(cudaMemcpyAsync(ex->out_block_h, ex->out_block_d, ex->out_block_bytes, cudaMemcpyDeviceToHost, s));
            continue;
        }
        CK(cudaMemcpyAsync(ex->n_h + f0, ex->n_d + f0, nf * sizeof(int), cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(ex->mono_h + f0, ex->mono_d + f0, nf * sizeof(int), cudaMemcpyDeviceToHost, s));
        if (direct) {
            if (keypoints_out)
                CK(cudaMemcpy2DAsync(keypoints_out + (size_t)f0 * capacity, (size_t)capacity * sizeof(vsg_keypoint), kd,
                                     (size_t)g.out_cap * sizeof(vsg_keypoint), (size_t)g.out_cap * sizeof(vsg_keypoint), nf,
                                     cudaMemcpyDeviceToHost, s));
            if (descriptors_out)
                CK(cudaMemcpy2DAsync(descriptors_out + (size_t)f0 * capacity * 32, (size_t)capacity * 32, dd,
                                     (size_t)g.out_cap * 32, (size_t)g.out_cap * 32, nf, cudaMemcpyDeviceToHost, s));
        } else {
            CK(cudaMemcpyAsync(ex->kps_h + (size_t)f0 * g.out_cap, kd, (size_t)nf * g.out_cap * sizeof(vsg_keypoint),
                               cudaMemcpyDeviceToHost, s));
            CK(cudaMemcpyAsync(ex->desc_h + (size_t)f0 * g.out_cap * 32, dd, (size_t)nf * g.out_cap * 32,
                               cudaMemcpyDeviceToHost, s));
        }
    }
    for (int k = 1; k < nstreams_used; ++k) CK(cudaStreamSynchronize(ex->aux[k - 1]));
    CK(cudaStreamSynchronize(ex->stream));
    vsg_status ret = VSG_OK;
    for (int f = 0; f < nframes; ++f) {
        const int n = ex->n_h[f];
        if (n_out) n_out[f] = n;
        if (mono_index_out) mono_index_out[f] = ex->mono_h[f];
        if (direct) continue;
        if (n > capacity) {
            set_error("vsg_extract_batch: frame %d has %d keypoints, capacity %d", f, n, capacity);
            ret = VSG_ERR_CAPACITY;
            continue;
        }
        if (keypoints_out)
            memcpy(keypoints_out + (size_t)f * capacity, ex->kps_h + (size_t)f * g.out_cap, (size_t)n * sizeof(vsg_keypoint));
        if (descriptors_out)
            memcpy(descriptors_out + (size_t)f * capacity * 32, ex->desc_h + (size_t)f * g.out_cap * 32, (size_t)n * 32);
    }
    return ret;
}

vsg_status vsg_extract_batch(vsg_extractor *ex, const uint8_t *images, int nframes, int width, int height, int pitch,
                             size_t frame_stride, int lap_x0, int lap_x1, vsg_keypoint *keypoints_out,
                             uint8_t *descriptors_out, int capacity, int *n_out, int *mono_index_out) {
    return extract_batch_host(ex, images, nframes, width, height, pitch, frame_stride, 1, 0, 0, lap_x0, lap_x1, keypoints_out,
                              descriptors_out, capacity, n_out, mono_index_out);
}

vsg_status vsg_extract_batch_color(vsg_extractor *ex, const uint8_t *images, int nframes, int width, int height, int pitch,
                                   size_t frame_stride, int channels, int r_first, int lap_x0, int lap_x1,
                                   vsg_keypoint *keypoints_out, uint8_t *descriptors_out, int capacity, int *n_out,
                                   int *mono_index_out) {
    if (channels != 3 && channels != 4) { set_error("vsg_extract_batch_color: channels must be 3 or 4"); return VSG_ERR_INVALID; }
    return extract_batch_host(ex, images, nframes, width, height, pitch, frame_stride, channels, r_first, 0, lap_x0, lap_x1,
                              keypoints_out, descriptors_out, capacity, n_out, mono_index_out);
}

vsg_status vsg_extractor_set_rectify_map(vsg_extractor *ex, int slot, const float *map_x, const float *map_y, int width,
                                         int height) {
    if (!ex || slot < 0 || slot > 1 || !map_x || !map_y || width <= 0 || height <= 0) {
        set_error("vsg_extractor_set_rectify_map: slot must be 0 or 1, maps non-null, size positive");
        return VSG_ERR_INVALID;
    }
    if (ex->rect_w != 0 && (ex->rect_w != width || ex->rect_h != height) && ex->rect_xy[1 - slot]) {
        set_error("vsg_extractor_set_rectify_map: both maps of a handle must have the same size (%dx%d vs %dx%d)", width, height,
                  ex->rect_w, ex->rect_h);
        return VSG_ERR_INVALID;
    }
    // cv::remap's fixed-point form of a CV_32FC1 map pair: sx = cvRound(x * INTER_TAB_SIZE), integer part saturated to short
    const size_t n = (size_t)width * height;
    std::vector<uint32_t> xy(n);
    std::vector<uint16_t> frac(n);
    auto sat_short = [](int v) { return v < -32768 ? -32768 : (v > 32767 ? 32767 : v); };
    for (size_t i = 0; i < n; ++i) {
        const int sx = cv_round(map_x[i] * 32.f), sy = cv_round(map_y[i] * 32.f);
        xy[i] = (uint32_t)(uint16_t)(short)sat_short(sx >> 5) | ((uint32_t)(uint16_t)(short)sat_short(sy >> 5) << 16);
        frac[i] = (uint16_t)(((sy & 31) << 5) | (sx & 31));
    }
    CK(cudaSetDevice(ex->device));
    CK(cudaStreamSynchronize(ex->stream));
    cudaFree(ex->rect_xy[slot]); cudaFree(ex->rect_frac[slot]);
    ex->rect_xy[slot] = nullptr; ex->rect_frac[slot] = nullptr;
    CK(cudaMalloc(&ex->rect_xy[slot], n * sizeof(uint32_t)));
    CK(cudaMalloc(&ex->rect_frac[slot], n * sizeof(uint16_t)));
    CK(cudaMemcpy(ex->rect_xy[slot], xy.data(), n * sizeof(uint32_t), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ex->rect_frac[slot], frac.data(), n * sizeof(uint16_t), cudaMemcpyHostToDevice));
    ex->rect_w = width; ex->rect_h = height;
    return VSG_OK;
}

vsg_status vsg_extract_batch_rectify(vsg_extractor *ex, const uint8_t *images, int nframes, int src_width, int src_height,
                                     int pitch, size_t frame_stride, int ncameras, int lap_x0, int lap_x1,
                                     vsg_keypoint *keypoints_out, uint8_t *descriptors_out, int capacity, int *n_out,
                                     int *mono_index_out) {
    if (!ex || ncameras < 1 || ncameras > 2 || !ex->rect_xy[0] || (ncameras == 2 && !ex->rect_xy[1])) {
        set_error("vsg_extract_batch_rectify: ncameras must be 1 or 2 and their maps set (vsg_extractor_set_rectify_map)");
        return VSG_ERR_INVALID;
    }
    return extract_batch_host(ex, images, nframes, src_width, src_height, pitch, frame_stride, 1, 0, ncameras, lap_x0, lap_x1,
                              keypoints_out, descriptors_out, capacity, n_out, mono_index_out);
}

vsg_status vsg_extract(vsg_extractor *ex, const uint8_t *image, int width, int height, int pitch, int lap_x0,
                       int lap_x1, vsg_keypoint *keypoints_out, uint8_t *descriptors_out, int capacity, int *n_out,
                       int *mono_index_out) {
    return vsg_extract_batch(ex, image, 1, width, height, pitch, (size_t)pitch * height, lap_x0, lap_x1, keypoints_out,
                             descriptors_out, capacity, n_out, mono_index_out);
}

vsg_status vsg_extract_batch_dev(vsg_extractor *ex, const uint8_t *images_dev, int nframes, int width, int height,
                                 int pitch, size_t frame_stride, int lap_x0, int lap_x1, vsg_keypoint *keypoints_dev,
                                 uint8_t *descriptors_dev, int capacity, int32_t *n_dev, int32_t *mono_dev) {
    if (!ex) return VSG_ERR_INVALID;
    if (!images_dev || width <= 0 || height <= 0 || nframes <= 0) return VSG_EMPTY_IMAGE;
    if (nframes > ex->max_batch || pitch < width || (pitch & 3) || ((uintptr_t)images_dev & 3) || (frame_stride & 3)) {
        set_error("vsg_extract_batch_dev: nframes > max_batch or unaligned device frames (need 4-byte aligned base/pitch/stride)");
        return VSG_ERR_INVALID;
    }
    CK(cudaSetDevice(ex->device));
    vsg_status st = configure_shape(ex, width, height);
    if (st != VSG_OK) return st;
    if (capacity < ex->g.out_cap) {
        set_error("vsg_extract_batch_dev: capacity %d < vsg_extractor_max_keypoints() = %d", capacity, ex->g.out_cap);
        return VSG_ERR_CAPACITY;
    }
    ex->lvl0_base = images_dev; ex->lvl0_pitch = pitch; ex->lvl0_stride = (int64_t)frame_stride; ex->last_nframes = nframes;
    ex->results_on_handle = false;
    return run_pipeline(ex, ex->stream, 0, images_dev, pitch, (int64_t)frame_stride, nframes, lap_x0, lap_x1, keypoints_dev,
                        descriptors_dev, capacity, n_dev, mono_dev);
}

vsg_status vsg_extractor_sync(vsg_extractor *ex) {
    if (!ex) return VSG_ERR_INVALID;
    CK(cudaStreamSynchronize(ex->stream));
    return VSG_OK;
}

void *vsg_extractor_stream(vsg_extractor *ex) { return ex ? (void *)ex->stream : nullptr; }

vsg_status vsg_extractor_profile(vsg_extractor *ex, int enable) {
    if (!ex) return VSG_ERR_INVALID;
    CK(cudaSetDevice(ex->device));
    CK(cudaStreamSynchronize(ex->stream));
    while (ex->ev_pending > 0) ex->harvest_one();
    ex->profile = enable != 0;
    for (int k = 0; k < VSG_NUM_STAGES; ++k) ex->stage_ms[k] = 0;
    ex->stage_runs = 0;
    return VSG_OK;
}

vsg_status vsg_extractor_stage_ms(vsg_extractor *ex, double *ms_out, int64_t *runs_out) {
    if (!ex) return VSG_ERR_INVALID;
    CK(cudaSetDevice(ex->device));
    CK(cudaStreamSynchronize(ex->stream));
    while (ex->ev_pending > 0) ex->harvest_one();
    for (int k = 0; k < VSG_NUM_STAGES; ++k) {
        if (ms_out) ms_out[k] = ex->stage_ms[k];
        ex->stage_ms[k] = 0;
    }
    if (runs_out) *runs_out = ex->stage_runs;
    ex->stage_runs = 0;
    return VSG_OK;
}

vsg_status vsg_pyramid_level_size(vsg_extractor *ex, int level, int *width, int *height) {
    if (!ex || ex->cur_w == 0 || level < 0 || level >= ex->g.nlevels) return VSG_ERR_INVALID;
    if (width) *width = ex->g.lv[level].w;
    if (height) *height = ex->g.lv[level].h;
    return VSG_OK;
}

static vsg_status download_plane(vsg_extractor *ex, const uint8_t *base, int frame, int level, bool allow_lvl0_ext,
                                 uint8_t *dst, int dst_pitch) {
    if (!ex || ex->cur_w == 0 || level < 0 || level >= ex->g.nlevels || frame < 0 || frame >= ex->last_nframes || !dst)
        return VSG_ERR_INVALID;
    const LevelGeom &L = ex->g.lv[level];
    const uint8_t *src = base + L.plane_offset + (int64_t)frame * L.plane_stride;
    int spitch = L.pitch;
    if (level == 0 && allow_lvl0_ext) { src = ex->lvl0_base + (int64_t)frame * ex->lvl0_stride; spitch = ex->lvl0_pitch; }
    CK(cudaSetDevice(ex->device));
    CK(cudaStreamSynchronize(ex->stream));
    CK(cudaMemcpy2D(dst, dst_pitch, src, spitch, L.w, L.h, cudaMemcpyDeviceToHost));
    return VSG_OK;
}

vsg_status vsg_pyramid_download(vsg_extractor *ex, int frame, int level, uint8_t *dst, int dst_pitch) {
    return download_plane(ex, ex ? ex->pyr : nullptr, frame, level, true, dst, dst_pitch);
}

vsg_status vsg_blurred_download(vsg_extractor *ex, int frame, int level, uint8_t *dst, int dst_pitch) {
    return download_plane(ex, ex ? ex->blur : nullptr, frame, level, false, dst, dst_pitch);
}

vsg_status vsg_candidates_download(vsg_extractor *ex, int frame, int level, int32_t *xys, int capacity, int *n_out) {
    if (!ex || ex->cur_w == 0 || level < 0 || level >= ex->g.nlevels || frame < 0 || frame >= ex->last_nframes)
        return VSG_ERR_INVALID;
    const FrameGeom &g = ex->g;
    const LevelGeom &L = g.lv[level];
    CK(cudaSetDevice(ex->device));
    CK(cudaStreamSynchronize(ex->stream));
    int n = 0;
    CK(cudaMemcpy(&n, ex->cand_count + frame * g.nlevels + level, sizeof(int), cudaMemcpyDeviceToHost));
    n = std::min(n, L.cand_cap);
    std::vector<Cand> c(n);
    CK(cudaMemcpy(c.data(), ex->cand + L.cand_offset + (int64_t)frame * g.cand_total, (size_t)n * sizeof(Cand),
                  cudaMemcpyDeviceToHost));
    // the device list is unordered; present it in the reference's order (cell-row-major, row-major inside a cell)
    auto key = [&](const Cand &a) {
        const int rx = a.x - kEdge, ry = a.y - kEdge;
        const int cx = rx / L.w_cell, cy = ry / L.h_cell;
        return ((int64_t)(cy * L.n_cols + cx) << 32) | ((int64_t)(ry - cy * L.h_cell) << 16) | (rx - cx * L.w_cell);
    };
    std::sort(c.begin(), c.end(), [&](const Cand &a, const Cand &b) { return key(a) < key(b); });
    if (n_out) *n_out = n;
    if (n > capacity) return VSG_ERR_CAPACITY;
    for (int i = 0; i < n; ++i) {
        xys[3 * i] = c[i].x - kBorderMin;
        xys[3 * i + 1] = c[i].y - kBorderMin;
        xys[3 * i + 2] = c[i].score;
    }
    return VSG_OK;
}

vsg_status vsg_level_keypoints_download(vsg_extractor *ex, int frame, int level, int32_t *xys, int capacity,
                                        int *n_out) {
    if (!ex || ex->cur_w == 0 || level < 0 || level >= ex->g.nlevels || frame < 0 || frame >= ex->last_nframes)
        return VSG_ERR_INVALID;
    const FrameGeom &g = ex->g;
    const LevelGeom &L = g.lv[level];
    CK(cudaSetDevice(ex->device));
    CK(cudaStreamSynchronize(ex->stream));
    int n = 0;
    CK(cudaMemcpy(&n, ex->level_kp_count + frame * g.nlevels + level, sizeof(int), cudaMemcpyDeviceToHost));
    std::vector<LevelKp> k(n);
    CK(cudaMemcpy(k.data(), ex->level_kps + (int64_t)frame * g.kp_total + L.kp_offset, (size_t)n * sizeof(LevelKp),
                  cudaMemcpyDeviceToHost));
    if (n_out) *n_out = n;
    if (n > capacity) return VSG_ERR_CAPACITY;
    for (int i = 0; i < n; ++i) {
        xys[3 * i] = k[i].x;
        xys[3 * i + 1] = k[i].y;
        xys[3 * i + 2] = k[i].score;
    }
    return VSG_OK;
}

}  // extern "C"
