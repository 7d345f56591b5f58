// capi.cu — host side of the C-ABI (include/plstvo.h): context, device buffers, work planning,
// chunked H2D / compute / D2H pipelining.  No CPU compute path exists in this library: without a CUDA
// device plstvo_create() fails with PLSTVO_E_NO_DEVICE and every other entry point needs a context.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"
#include "match_tc.cuh"

using namespace plstvo;

namespace {

struct DevBuf {
    void*  p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// Work plan + device storage of one batch of frame pairs (also the body of PlDeviceBatch)
struct Workspace {
    int B = 0;
    PlCamera cam{};
    PlConfig cfg{};
    bool has_priors = false;
    bool have_level = false;   // prev->ls_level supplied (null = level 0 everywhere)
    bool planned = false, planned_features = false;   // plan cache (ws_prepare)
    int sm_planned = 0;
    // host copies of the offsets
    std::vector<int32_t> p_off1, p_off2, l_off1, l_off2;
    // plan
    std::vector<MatchProblem> problems;   // [2B]: points, lines
    int cap_pt = 0, cap_ls = 0, sort_cap = 1, max_n2 = 0;
    bool feat_in_smem = true;
    // device storage
    DevBuf d_poff1, d_poff2, d_loff1, d_loff2;
    DevBuf d_pdesc1, d_pdesc2, d_ldesc1, d_ldesc2;
    DevBuf d_ptP, d_pts2, d_ptpl;                                      // prev P, prev sigma2, curr pl
    DevBuf d_lssP, d_lseP, d_lsspl, d_lsepl, d_lss2, d_lslev, d_lsle;  // prev ...; curr le
    DevBuf d_priors, d_results, d_m12p, d_m12l, d_inlp, d_inll;
    DevBuf d_rowpart, d_colpart, d_problems, d_feat;
    DevBuf d_phase;   // debug phase timers (PLSTVO_PHASE_DEBUG)
    // K1 on the tensor cores (match_tc.cu): expanded operands, per-block value partials, work items
    std::vector<TcProblem> tc_problems;   // [2B], parallel to `problems`
    std::vector<TcSide> tc_sides;         // [4B]: queries, trains of every problem
    std::vector<TcItem> tc_items[2];      // work items of the point problems (long) and of the line problems (short)
    std::vector<int32_t> item_start[2];   // [B+1] first work item of each pair in either list
    int tc_max_tiles = 0;
    DevBuf d_tcprob, d_tcsides, d_tcitems[2], d_exp, d_rowp, d_colp, d_sched;
    DevBuf d_stream;       // arena of the streamed solver (frames too large for K2's shared memory)
    bool use_stream = false;
    size_t feat_stride = 0;
    void release() {
        DevBuf* all[] = {&d_poff1, &d_poff2, &d_loff1, &d_loff2, &d_pdesc1, &d_pdesc2, &d_ldesc1, &d_ldesc2,
                         &d_ptP, &d_pts2, &d_ptpl, &d_lssP, &d_lseP, &d_lsspl, &d_lsepl, &d_lss2, &d_lslev,
                         &d_lsle, &d_priors, &d_results, &d_m12p, &d_m12l, &d_inlp, &d_inll, &d_rowpart,
                         &d_colpart, &d_problems, &d_feat, &d_phase, &d_tcprob, &d_tcsides, &d_tcitems[0],
                         &d_tcitems[1], &d_exp, &d_rowp, &d_colp, &d_sched, &d_stream};
        for (DevBuf* b : all) b->release();
    }
};

}  // namespace

struct PlContext {
    std::recursive_mutex mu;   // entry points serialise on it: one context may be shared by the caller's threads
    int device = 0;
    int sm_count = 0;
    size_t smem_optin = 0;
    cudaStream_t s_main = nullptr, s_alt = nullptr, s_h2d = nullptr, s_d2h = nullptr;
    std::vector<cudaEvent_t> events;
    size_t next_event = 0;
    std::string err;
    int64_t launches = 0;
    Workspace ws;          // reused by the host-buffer entry points
    Workspace ws_async[2]; // double-buffered workspaces of plstvo_track_batch_async
    cudaEvent_t slot_done[2] = {nullptr, nullptr};
    bool slot_busy[2] = {false, false};
    int next_slot = 0;
    DevBuf scratch;        // misc (popc bench, L2 flush)
    DevBuf gn_in[8], gn_out[4];
    // per-entry-point device arenas (context-owned: a process may hold one context per GPU)
    DevBuf arena_grid, arena_lift_pt, arena_lift_ls, arena_stereo;
    DevBuf arena_track_stereo[3];   // [0]: blocking calls, [1 + slot]: plstvo_track_stereo_*_async
    DevBuf gs_in[13], gs_rec_pt, gs_rec_ls;   // resident inputs / packed records of the streamed evaluator
    // pinned host scratch (small tables and counters that must not block the enqueueing thread), same indexing as the arenas
    void* h_staging[3] = {nullptr, nullptr, nullptr};
    size_t h_staging_bytes[3] = {0, 0, 0};
    cudaError_t staging(int k, size_t bytes) {
        if (bytes <= h_staging_bytes[k]) return cudaSuccess;
        if (h_staging[k]) cudaFreeHost(h_staging[k]);
        h_staging[k] = nullptr;
        h_staging_bytes[k] = 0;
        cudaError_t e = cudaMallocHost(&h_staging[k], bytes);
        if (e == cudaSuccess) h_staging_bytes[k] = bytes;
        return e;
    }
};

struct PlDeviceBatch {
    Workspace ws;
};

namespace {

#define CK(ctx, call)                                                                            \
    do {                                                                                         \
        cudaError_t e__ = (call);                                                                \
        if (e__ != cudaSuccess) {                                                                \
            char buf__[512];                                                                     \
            snprintf(buf__, sizeof(buf__), "%s:%d: %s -> %s", __FILE__, __LINE__, #call,         \
                     cudaGetErrorString(e__));                                                   \
            (ctx)->err = buf__;                                                                  \
            return PLSTVO_E_CUDA;                                                                \
        }                                                                                        \
    } while (0)

#define LOCK(ctx) std::lock_guard<std::recursive_mutex> lock__((ctx)->mu)

int fail(PlContext* ctx, int code, const char* msg) {
    if (ctx) ctx->err = msg;
    return code;
}

// Cross-stream ordering events.  Each one is recorded and immediately waited on by the enqueuing host code, so a ring
// can be recycled while earlier work is still in flight (a wait captures the record that preceded it).
cudaEvent_t next_event(PlContext* ctx) {
    constexpr size_t RING = 512;
    if (ctx->events.size() < RING) {
        cudaEvent_t e;
        cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
        ctx->events.push_back(e);
        return e;
    }
    return ctx->events[ctx->next_event++ % RING];
}

int pow2_ceil_host(int n) {
    int m = 1;
    while (m < n) m <<= 1;
    return m;
}


// Which solver a batch takes.  K2 (one fp64 CTA per pair, lists in shared memory) has the lower latency and follows the
// reference to rounding; the streamed solver (fp32 per-feature arithmetic, fp64 sums / algebra / outlier statistics, close stop
// tests re-decided in fp64) has the higher throughput once a batch is more than one wave of K2 CTAs, and is the only form for
// lists that do not fit K2's shared memory.  Default: streamed when the lists do not fit, or when the batch has more pairs than
// the device has SMs.  PLSTVO_STREAM_SOLVE=1: always streamed (tests on small frames); =0: never (K2, lists in global scratch
// if need be).
int stream_mode() {
    static const int m = [] {
        const char* v = getenv("PLSTVO_STREAM_SOLVE");
        return v ? atoi(v) : -1;
    }();
    return m;
}

// carves the streamed solver's buffers for B problems out of one arena; slots = record slots (prev-frame features in track
// mode, list entries in explicit mode)
int stream_bufs_prepare(PlContext* ctx, DevBuf& arena, int B, size_t slots_pt, size_t slots_ls, StreamBufs* sb) {
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const size_t o_rp = take((slots_pt + 512) * 2 * sizeof(float4)), o_rl = take((slots_ls + 256) * 4 * sizeof(float4));
    const size_t o_cp = take((size_t)B * 4), o_cl = take((size_t)B * 4), o_dt = take((size_t)B * 16 * 8), o_ac = take((size_t)B * 4);
    const size_t o_ctl = take((size_t)B * sizeof(StreamCtl));
    const size_t o_fp = take(slots_pt + 16), o_fl = take(slots_ls + 16), o_mp = take((slots_pt + 16) * 2), o_ml = take((slots_ls + 16) * 2);
    const size_t o_q = take((size_t)B * 2 * 4 + 16);
    CK(ctx, arena.ensure(off));
    uint8_t* b = arena.as<uint8_t>();
    sb->rec_pt = reinterpret_cast<float4*>(b + o_rp);
    sb->rec_ls = reinterpret_cast<float4*>(b + o_rl);
    sb->cnt_pt = reinterpret_cast<int32_t*>(b + o_cp);
    sb->cnt_ls = reinterpret_cast<int32_t*>(b + o_cl);
    sb->DT = reinterpret_cast<double*>(b + o_dt);
    sb->active = reinterpret_cast<int32_t*>(b + o_ac);
    sb->ctl = reinterpret_cast<StreamCtl*>(b + o_ctl);
    sb->queue = reinterpret_cast<int32_t*>(b + o_q);
    sb->flag_pt = b + o_fp;
    sb->flag_ls = b + o_fl;
    sb->midx_pt = reinterpret_cast<uint16_t*>(b + o_mp);
    sb->midx_ls = reinterpret_cast<uint16_t*>(b + o_ml);
    sb->sm_count = ctx->sm_count;
    return 0;
}

// the per-problem arrays of a chunk of pairs starting at p0 (record / flag arrays are indexed by absolute slots)
StreamBufs stream_bufs_at(const StreamBufs& sb, int p0) {
    StreamBufs r = sb;
    r.cnt_pt += p0; r.cnt_ls += p0; r.DT += (size_t)p0 * 16; r.active += p0; r.ctl += p0;
    r.queue += 2 * (size_t)p0;   // a chunk starts at a distinct pair: its two queue words are its own
    return r;
}

// ---- planning -------------------------------------------------------------------------------------
void plan_problem(MatchProblem& pr, int n1, int n2, bool enabled, float nnr, int best_lr) {
    pr.n1 = n1;
    pr.n2 = n2;
    pr.nnr = nnr;
    pr.best_lr = best_lr;
    pr.enabled = (enabled && n1 > 0 && n2 > 0) ? 1 : 0;   // src/stereoFrameHandler.cpp:137-138, :160-161
}

int validate_frames(PlContext* ctx, const PlFrameBatch* prev, const PlFrameBatch* curr, bool need_features) {
    if (!prev || !curr) return fail(ctx, PLSTVO_E_INVALID, "null frame batch");
    if (prev->B != curr->B) return fail(ctx, PLSTVO_E_SIZE, "prev and curr hold a different number of frames");
    if (prev->B < 0) return fail(ctx, PLSTVO_E_INVALID, "negative batch size");
    if (prev->B == 0) return 0;
    if (!prev->pt_off || !prev->ls_off || !curr->pt_off || !curr->ls_off)
        return fail(ctx, PLSTVO_E_INVALID, "null offsets");
    if (prev->pt_off[0] || prev->ls_off[0] || curr->pt_off[0] || curr->ls_off[0])
        return fail(ctx, PLSTVO_E_INVALID, "offsets must start at 0");
    for (int p = 0; p < prev->B; ++p) {
        const int n[4] = {prev->pt_off[p + 1] - prev->pt_off[p], curr->pt_off[p + 1] - curr->pt_off[p],
                          prev->ls_off[p + 1] - prev->ls_off[p], curr->ls_off[p + 1] - curr->ls_off[p]};
        for (int k = 0; k < 4; ++k) {
            if (n[k] < 0) return fail(ctx, PLSTVO_E_INVALID, "offsets are not non-decreasing");
            if (n[k] > PLSTVO_MAX_FEATURES) return fail(ctx, PLSTVO_E_TOO_LARGE, "more than 65535 features in a frame");
        }
    }
    const int np1 = prev->pt_off[prev->B], np2 = curr->pt_off[curr->B];
    const int nl1 = prev->ls_off[prev->B], nl2 = curr->ls_off[curr->B];
    if ((np1 && !prev->pdesc) || (np2 && !curr->pdesc) || (nl1 && !prev->ldesc) || (nl2 && !curr->ldesc))
        return fail(ctx, PLSTVO_E_INVALID, "null descriptor matrix");
    if (need_features) {
        if (np1 && (!prev->pt_P || !prev->pt_sigma2)) return fail(ctx, PLSTVO_E_INVALID, "prev point arrays missing");
        if (np2 && !curr->pt_pl) return fail(ctx, PLSTVO_E_INVALID, "curr pt_pl missing");
        if (nl1 && (!prev->ls_sP || !prev->ls_eP || !prev->ls_spl || !prev->ls_epl || !prev->ls_sigma2))
            return fail(ctx, PLSTVO_E_INVALID, "prev line arrays missing");
        if (nl2 && !curr->ls_le) return fail(ctx, PLSTVO_E_INVALID, "curr ls_le missing");
    }
    return 0;
}

// Builds the plan of a batch of pairs and sizes every device buffer.  `with_features` = track mode.
int ws_prepare(PlContext* ctx, Workspace& ws, const PlCamera* cam, const PlConfig* cfg, const PlFrameBatch* prev,
               const PlFrameBatch* curr, bool with_features, bool has_priors) {
    const int B = prev->B;
    // Same shapes and matching parameters as the previous call on this workspace (a video stream, a benchmark loop):
    // the plan, the partial buffers and their device copies are still valid — skip the rebuild and its uploads.
    if (ws.planned && ws.B == B && ws.planned_features == with_features && ws.sm_planned == ctx->sm_count &&
        ws.cfg.has_points == cfg->has_points && ws.cfg.has_lines == cfg->has_lines &&
        ws.cfg.best_lr_matches == cfg->best_lr_matches && ws.cfg.min_ratio_12_p == cfg->min_ratio_12_p &&
        (ws.cfg.solver_mode != 0) == (cfg->solver_mode != 0) &&
        ws.cfg.min_ratio_12_l == cfg->min_ratio_12_l && (int)ws.p_off1.size() == B + 1 &&
        !memcmp(ws.p_off1.data(), prev->pt_off, (size_t)(B + 1) * 4) &&
        !memcmp(ws.p_off2.data(), curr->pt_off, (size_t)(B + 1) * 4) &&
        !memcmp(ws.l_off1.data(), prev->ls_off, (size_t)(B + 1) * 4) &&
        !memcmp(ws.l_off2.data(), curr->ls_off, (size_t)(B + 1) * 4)) {
        if (cam) ws.cam = *cam;
        ws.cfg = *cfg;
        ws.has_priors = has_priors;
        return 0;
    }
    ws.planned = false;
    ws.B = B;
    if (cam) ws.cam = *cam;
    ws.cfg = *cfg;
    ws.has_priors = has_priors;
    ws.p_off1.assign(prev->pt_off, prev->pt_off + B + 1);
    ws.p_off2.assign(curr->pt_off, curr->pt_off + B + 1);
    ws.l_off1.assign(prev->ls_off, prev->ls_off + B + 1);
    ws.l_off2.assign(curr->ls_off, curr->ls_off + B + 1);
    const size_t np1 = ws.p_off1[B], np2 = ws.p_off2[B], nl1 = ws.l_off1[B], nl2 = ws.l_off2[B];

    ws.problems.assign((size_t)2 * B, MatchProblem{});
    ws.cap_pt = ws.cap_ls = 0;
    ws.max_n2 = 0;
    size_t row_elems = 0, col_elems = 0, exp_tiles = 0, rowp_elems = 0, colp_elems = 0;
    ws.tc_problems.assign((size_t)2 * B, TcProblem{});
    ws.tc_sides.assign((size_t)4 * B, TcSide{});
    for (int k = 0; k < 2; ++k) {
        ws.tc_items[k].clear();
        ws.item_start[k].assign((size_t)B + 1, 0);
    }
    ws.tc_max_tiles = 0;
    const float nnr_p = (float)cfg->min_ratio_12_p, nnr_l = (float)cfg->min_ratio_12_l;   // double -> float at the call
    for (int p = 0; p < B; ++p) {
        ws.item_start[0][p] = (int32_t)ws.tc_items[0].size();
        ws.item_start[1][p] = (int32_t)ws.tc_items[1].size();
        for (int type = 0; type < 2; ++type) {
            MatchProblem& pr = ws.problems[(size_t)2 * p + type];
            const int n1 = type ? ws.l_off1[p + 1] - ws.l_off1[p] : ws.p_off1[p + 1] - ws.p_off1[p];
            const int n2 = type ? ws.l_off2[p + 1] - ws.l_off2[p] : ws.p_off2[p + 1] - ws.p_off2[p];
            plan_problem(pr, n1, n2, type ? cfg->has_lines != 0 : cfg->has_points != 0, type ? nnr_l : nnr_p,
                         cfg->best_lr_matches != 0);
            // operands and partials as element / tile indices first, fixed up after allocation
            const int t1 = pr.enabled ? (n1 + TC_ROWS - 1) / TC_ROWS : 0, t2 = pr.enabled ? (n2 + TC_ROWS - 1) / TC_ROWS : 0;
            TcProblem& tp = ws.tc_problems[(size_t)2 * p + type];
            tp.n1 = n1;
            tp.n2 = n2;
            tp.xe = reinterpret_cast<const uint8_t*>(exp_tiles);
            tp.ye = reinterpret_cast<const uint8_t*>(exp_tiles + t1);
            tp.rowp = reinterpret_cast<uint32_t*>(rowp_elems);
            tp.colp = reinterpret_cast<uint32_t*>(colp_elems);
            ws.tc_sides[(size_t)4 * p + 2 * type] = TcSide{nullptr, pr.enabled ? n1 : 0, nullptr};
            ws.tc_sides[(size_t)4 * p + 2 * type + 1] = TcSide{nullptr, pr.enabled ? n2 : 0, nullptr};
            exp_tiles += (size_t)t1 + t2;
            rowp_elems += (size_t)(pr.enabled ? (n2 + TC_CW - 1) / TC_CW : 0) * n1;
            colp_elems += (size_t)(pr.enabled ? n2 : 0);
            ws.tc_max_tiles = std::max(ws.tc_max_tiles, std::max(t1, t2));
            for (int yb = 0; yb < (t2 + 1) / 2; ++yb) ws.tc_items[type].push_back(TcItem{2 * p + type, yb});
            // one merged key pair per row and per column (tc_resolve_kernel), also as element indices first
            pr.rowpart = reinterpret_cast<uint2*>(row_elems);
            pr.colpart = reinterpret_cast<uint2*>(col_elems);
            row_elems += (size_t)(pr.enabled ? n1 : 0);
            col_elems += (size_t)(pr.enabled ? n2 : 0);
            ws.max_n2 = std::max(ws.max_n2, n2);
            if (type == 0) ws.cap_pt = std::max(ws.cap_pt, n1);
            else ws.cap_ls = std::max(ws.cap_ls, n1);
        }
    }
    ws.item_start[0][B] = (int32_t)ws.tc_items[0].size();
    ws.item_start[1][B] = (int32_t)ws.tc_items[1].size();
    ws.cap_pt = std::max(ws.cap_pt, 1);
    ws.cap_ls = std::max(ws.cap_ls, 1);
    // at least 32: the outlier statistics sort max(n, 32) padded entries (solve.cu: remove_outliers)
    ws.sort_cap = pow2_ceil_host(std::max(32, std::max(std::max(ws.cap_pt, ws.cap_ls), (ws.max_n2 + 1) / 2)));
    // matched lists live in shared memory when they fit (C2: 152 KB), else in a global scratch slice (C5)
    static const bool no_smem = getenv("PLSTVO_K2_FEAT_GLOBAL") != nullptr;
    ws.feat_in_smem = !no_smem && k2_smem_bytes(ws.cap_pt, ws.cap_ls, ws.sort_cap, true) <= ctx->smem_optin;
    // the per-pair solver's limits only apply when it runs (track mode): matching-only calls take any frame up to
    // PLSTVO_MAX_FEATURES rows
    if (with_features && !ws.feat_in_smem && k2_smem_bytes(ws.cap_pt, ws.cap_ls, ws.sort_cap, false) > ctx->smem_optin)
        return fail(ctx, PLSTVO_E_TOO_LARGE, "frame too large for the per-pair solver's shared memory");

    // --- device storage ---
    CK(ctx, ws.d_pdesc1.ensure(np1 * 32));
    CK(ctx, ws.d_pdesc2.ensure(np2 * 32));
    CK(ctx, ws.d_ldesc1.ensure(nl1 * 32));
    CK(ctx, ws.d_ldesc2.ensure(nl2 * 32));
    CK(ctx, ws.d_m12p.ensure(np1 * 4));
    CK(ctx, ws.d_m12l.ensure(nl1 * 4));
    CK(ctx, ws.d_rowpart.ensure(row_elems * sizeof(uint2)));
    CK(ctx, ws.d_colpart.ensure(col_elems * sizeof(uint2)));
    CK(ctx, ws.d_problems.ensure(ws.problems.size() * sizeof(MatchProblem)));
    CK(ctx, ws.d_exp.ensure(exp_tiles * TC_TILE_BYTES + 1024));
    CK(ctx, ws.d_rowp.ensure(rowp_elems * sizeof(uint32_t)));
    CK(ctx, ws.d_colp.ensure(colp_elems * sizeof(uint32_t)));
    CK(ctx, ws.d_tcprob.ensure(ws.tc_problems.size() * sizeof(TcProblem)));
    CK(ctx, ws.d_tcsides.ensure(ws.tc_sides.size() * sizeof(TcSide)));
    for (int k = 0; k < 2; ++k) CK(ctx, ws.d_tcitems[k].ensure(ws.tc_items[k].size() * sizeof(TcItem)));
    if (!ws.d_sched.p) {   // scheduler words of the persistent matcher: one pair per compute stream, self re-arming
        CK(ctx, ws.d_sched.ensure(64));
        CK(ctx, cudaMemsetAsync(ws.d_sched.p, 0, 64, ctx->s_h2d));
    }
    if (with_features) {
        CK(ctx, ws.d_poff1.ensure((B + 1) * 4));
        CK(ctx, ws.d_poff2.ensure((B + 1) * 4));
        CK(ctx, ws.d_loff1.ensure((B + 1) * 4));
        CK(ctx, ws.d_loff2.ensure((B + 1) * 4));
        CK(ctx, ws.d_ptP.ensure(np1 * 24));
        CK(ctx, ws.d_pts2.ensure(np1 * 8));
        CK(ctx, ws.d_ptpl.ensure(np2 * 16));
        CK(ctx, ws.d_lssP.ensure(nl1 * 24));
        CK(ctx, ws.d_lseP.ensure(nl1 * 24));
        CK(ctx, ws.d_lsspl.ensure(nl1 * 16));
        CK(ctx, ws.d_lsepl.ensure(nl1 * 16));
        CK(ctx, ws.d_lss2.ensure(nl1 * 8));
        CK(ctx, ws.d_lslev.ensure(nl1 * 4));
        CK(ctx, ws.d_lsle.ensure(nl2 * 24));
        CK(ctx, ws.d_priors.ensure((size_t)B * sizeof(PlPrior)));
        CK(ctx, ws.d_results.ensure((size_t)B * sizeof(PlPoseResult)));
        CK(ctx, ws.d_inlp.ensure(np1));
        CK(ctx, ws.d_inll.ensure(nl1));
        // (the robust main solver, solver_mode != 0, is K2-only: the streamed form would hand every problem back)
        ws.use_stream = stream_mode() == 1 ||
                        (stream_mode() != 0 && (!ws.feat_in_smem || (B > ctx->sm_count && cfg->solver_mode == 0)));
        if (!ws.feat_in_smem || ws.use_stream) {
            ws.feat_stride = k2_feat_stride(ws.cap_pt, ws.cap_ls);
            CK(ctx, ws.d_feat.ensure((size_t)B * ws.feat_stride * sizeof(double)));
        }
    }
    // --- fix up pointers, upload the plan ---
    for (int p = 0; p < B; ++p)
        for (int type = 0; type < 2; ++type) {
            MatchProblem& pr = ws.problems[(size_t)2 * p + type];
            pr.rowpart = ws.d_rowpart.as<uint2>() + reinterpret_cast<size_t>(pr.rowpart);
            pr.colpart = ws.d_colpart.as<uint2>() + reinterpret_cast<size_t>(pr.colpart);
            if (type == 0) {
                pr.d1 = ws.d_pdesc1.as<uint8_t>() + (size_t)ws.p_off1[p] * 32;
                pr.d2 = ws.d_pdesc2.as<uint8_t>() + (size_t)ws.p_off2[p] * 32;
                pr.m12 = ws.d_m12p.as<int32_t>() + ws.p_off1[p];
            } else {
                pr.d1 = ws.d_ldesc1.as<uint8_t>() + (size_t)ws.l_off1[p] * 32;
                pr.d2 = ws.d_ldesc2.as<uint8_t>() + (size_t)ws.l_off2[p] * 32;
                pr.m12 = ws.d_m12l.as<int32_t>() + ws.l_off1[p];
            }
            TcProblem& tp = ws.tc_problems[(size_t)2 * p + type];
            uint8_t* ebase = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws.d_exp.p) + 1023) & ~(uintptr_t)1023);
            uint8_t* xe = ebase + reinterpret_cast<size_t>(tp.xe) * TC_TILE_BYTES;
            uint8_t* ye = ebase + reinterpret_cast<size_t>(tp.ye) * TC_TILE_BYTES;
            tp.xe = xe;
            tp.ye = ye;
            tp.rowp = ws.d_rowp.as<uint32_t>() + reinterpret_cast<size_t>(tp.rowp);
            tp.colp = ws.d_colp.as<uint32_t>() + reinterpret_cast<size_t>(tp.colp);
            ws.tc_sides[(size_t)4 * p + 2 * type].src = pr.d1;
            ws.tc_sides[(size_t)4 * p + 2 * type].dst = xe;
            ws.tc_sides[(size_t)4 * p + 2 * type + 1].src = pr.d2;
            ws.tc_sides[(size_t)4 * p + 2 * type + 1].dst = ye;
        }
    cudaStream_t s = ctx->s_h2d;
    if (!ws.tc_problems.empty()) {
        CK(ctx, cudaMemcpyAsync(ws.d_tcprob.p, ws.tc_problems.data(), ws.tc_problems.size() * sizeof(TcProblem),
                                cudaMemcpyHostToDevice, s));
        CK(ctx, cudaMemcpyAsync(ws.d_tcsides.p, ws.tc_sides.data(), ws.tc_sides.size() * sizeof(TcSide),
                                cudaMemcpyHostToDevice, s));
        for (int k = 0; k < 2; ++k)
            if (!ws.tc_items[k].empty())
                CK(ctx, cudaMemcpyAsync(ws.d_tcitems[k].p, ws.tc_items[k].data(), ws.tc_items[k].size() * sizeof(TcItem),
                                        cudaMemcpyHostToDevice, s));
    }
    if (!ws.problems.empty())
        CK(ctx, cudaMemcpyAsync(ws.d_problems.p, ws.problems.data(), ws.problems.size() * sizeof(MatchProblem),
                                cudaMemcpyHostToDevice, s));
    if (with_features) {
        CK(ctx, cudaMemcpyAsync(ws.d_poff1.p, ws.p_off1.data(), (B + 1) * 4, cudaMemcpyHostToDevice, s));
        CK(ctx, cudaMemcpyAsync(ws.d_poff2.p, ws.p_off2.data(), (B + 1) * 4, cudaMemcpyHostToDevice, s));
        CK(ctx, cudaMemcpyAsync(ws.d_loff1.p, ws.l_off1.data(), (B + 1) * 4, cudaMemcpyHostToDevice, s));
        CK(ctx, cudaMemcpyAsync(ws.d_loff2.p, ws.l_off2.data(), (B + 1) * 4, cudaMemcpyHostToDevice, s));
    }
    ws.planned = true;
    ws.planned_features = with_features;
    ws.sm_planned = ctx->sm_count;
    return 0;
}

#define H2D(ctx, dst, src, elem_bytes, first, count, stream)                                                 \
    do {                                                                                                     \
        if ((count) > 0 && (src) != nullptr)                                                                 \
            CK(ctx, cudaMemcpyAsync((dst).as<uint8_t>() + (size_t)(first) * (elem_bytes),                    \
                                    reinterpret_cast<const uint8_t*>(src) + (size_t)(first) * (elem_bytes),  \
                                    (size_t)(count) * (elem_bytes), cudaMemcpyHostToDevice, stream));        \
    } while (0)

// descriptors (+ features when with_features) of pairs [p0, p1) host -> device
int ws_upload_range(PlContext* ctx, Workspace& ws, const PlFrameBatch* prev, const PlFrameBatch* curr,
                    const PlPrior* priors, int p0, int p1, bool with_features, cudaStream_t s) {
    const int a = ws.p_off1[p0], an = ws.p_off1[p1] - a, b = ws.p_off2[p0], bn = ws.p_off2[p1] - b;
    const int c = ws.l_off1[p0], cn = ws.l_off1[p1] - c, d = ws.l_off2[p0], dn = ws.l_off2[p1] - d;
    H2D(ctx, ws.d_pdesc1, prev->pdesc, 32, a, an, s);
    H2D(ctx, ws.d_pdesc2, curr->pdesc, 32, b, bn, s);
    H2D(ctx, ws.d_ldesc1, prev->ldesc, 32, c, cn, s);
    H2D(ctx, ws.d_ldesc2, curr->ldesc, 32, d, dn, s);
    if (with_features) {
        H2D(ctx, ws.d_ptP, prev->pt_P, 24, a, an, s);
        H2D(ctx, ws.d_pts2, prev->pt_sigma2, 8, a, an, s);
        H2D(ctx, ws.d_ptpl, curr->pt_pl, 16, b, bn, s);
        H2D(ctx, ws.d_lssP, prev->ls_sP, 24, c, cn, s);
        H2D(ctx, ws.d_lseP, prev->ls_eP, 24, c, cn, s);
        H2D(ctx, ws.d_lsspl, prev->ls_spl, 16, c, cn, s);
        H2D(ctx, ws.d_lsepl, prev->ls_epl, 16, c, cn, s);
        H2D(ctx, ws.d_lss2, prev->ls_sigma2, 8, c, cn, s);
        H2D(ctx, ws.d_lslev, prev->ls_level, 4, c, cn, s);
        H2D(ctx, ws.d_lsle, curr->ls_le, 24, d, dn, s);
        if (priors) H2D(ctx, ws.d_priors, priors, sizeof(PlPrior), p0, p1 - p0, s);
    }
    return 0;
}

int ws_launch_match(PlContext* ctx, Workspace& ws, int p0, int p1, cudaStream_t s, cudaEvent_t* marks = nullptr) {
    const int a0 = ws.item_start[0][p0], a1 = ws.item_start[0][p1], b0 = ws.item_start[1][p0], b1 = ws.item_start[1][p1];
    if (a1 > a0 || b1 > b0) {
        CK(ctx, launch_tc_expand(ws.d_tcsides.as<TcSide>() + (size_t)4 * p0, 4 * (p1 - p0), ws.tc_max_tiles, s));
        if (marks) CK(ctx, cudaEventRecord(marks[0], s));
        // launches on the two compute streams may overlap: each has its own pair of scheduler words
        int* sched = ws.d_sched.as<int>() + (s == ctx->s_alt ? 8 : 0);
        CK(ctx, launch_tc_hamming(ws.d_tcprob.as<TcProblem>(), ws.d_tcitems[0].as<TcItem>() + a0, a1 - a0,
                                  ws.d_tcitems[1].as<TcItem>() + b0, b1 - b0, sched, ctx->sm_count, nullptr, s));
        if (marks) CK(ctx, cudaEventRecord(marks[1], s));
        CK(ctx, launch_tc_resolve(ws.d_problems.as<MatchProblem>() + (size_t)2 * p0, ws.d_tcprob.as<TcProblem>() + (size_t)2 * p0,
                                  2 * (p1 - p0), 4, s));
        ctx->launches += 3;
    }
    return 0;
}

int ws_launch_solve(PlContext* ctx, Workspace& ws, int p0, int p1, bool have_level, cudaStream_t s, cudaEvent_t* marks = nullptr) {
    if (p1 <= p0) return 0;
    SolveParams prm{};
    prm.cam = ws.cam;
    prm.cfg = ws.cfg;
    prm.mode = 0;
    prm.first_pair = p0;
    prm.prev = FrameDev{ws.d_poff1.as<int32_t>(), ws.d_loff1.as<int32_t>(), nullptr, nullptr,
                        ws.d_ptP.as<double>(), nullptr, ws.d_pts2.as<double>(), ws.d_lssP.as<double>(),
                        ws.d_lseP.as<double>(), nullptr, ws.d_lsspl.as<double>(), ws.d_lsepl.as<double>(),
                        ws.d_lss2.as<double>(), have_level ? ws.d_lslev.as<int32_t>() : nullptr};
    prm.curr = FrameDev{ws.d_poff2.as<int32_t>(), ws.d_loff2.as<int32_t>(), nullptr, nullptr, nullptr,
                        ws.d_ptpl.as<double>(), nullptr, nullptr, nullptr, ws.d_lsle.as<double>(), nullptr,
                        nullptr, nullptr, nullptr};
    prm.problems = ws.d_problems.as<MatchProblem>();
    prm.priors = ws.has_priors ? ws.d_priors.as<PlPrior>() : nullptr;
    prm.results = ws.d_results.as<PlPoseResult>();
    prm.inlier_pt = ws.d_inlp.as<uint8_t>();
    prm.inlier_ls = ws.d_inll.as<uint8_t>();
    prm.feat_scratch = ws.feat_in_smem ? nullptr : ws.d_feat.as<double>() + (size_t)p0 * ws.feat_stride;
    prm.feat_scratch_stride = ws.feat_stride;
    prm.cap_pt = ws.cap_pt;
    prm.cap_ls = ws.cap_ls;
    prm.sort_cap = ws.sort_cap;
    prm.feat_in_smem = ws.feat_in_smem ? 1 : 0;
    prm.phase_cycles = ws.d_phase.as<long long>();
    if (ws.use_stream) {
        StreamBufs sb;
        int rc = stream_bufs_prepare(ctx, ws.d_stream, ws.B, (size_t)ws.p_off1[ws.B], (size_t)ws.l_off1[ws.B], &sb);
        if (rc) return rc;
        prm.feat_scratch = ws.d_feat.as<double>() + (size_t)p0 * ws.feat_stride;
        prm.feat_in_smem = 0;
        int nl = 0;
        CK(ctx, launch_stream_solve(prm, p1 - p0, stream_bufs_at(sb, p0), s, &nl, marks));
        ctx->launches += nl;
        return 0;
    }
    if (marks)   // fused kernel: list building, both GN stages and the outlier pass are inside K2
        for (int k = 0; k < 4; ++k) CK(ctx, cudaEventRecord(marks[k], s));
    CK(ctx, launch_track_solve(prm, p1 - p0, s));
    ctx->launches++;
    return 0;
}

#define D2H(ctx, dst, src, elem_bytes, first, count, stream)                                                 \
    do {                                                                                                     \
        if ((count) > 0 && (dst) != nullptr)                                                                 \
            CK(ctx, cudaMemcpyAsync(reinterpret_cast<uint8_t*>(dst) + (size_t)(first) * (elem_bytes),        \
                                    (src).as<uint8_t>() + (size_t)(first) * (elem_bytes),                    \
                                    (size_t)(count) * (elem_bytes), cudaMemcpyDeviceToHost, stream));        \
    } while (0)

int ws_download_range(PlContext* ctx, Workspace& ws, int p0, int p1, PlPoseResult* results, int32_t* m12_pt,
                      int32_t* m12_ls, uint8_t* inl_pt, uint8_t* inl_ls, cudaStream_t s) {
    const int a = ws.p_off1[p0], an = ws.p_off1[p1] - a, c = ws.l_off1[p0], cn = ws.l_off1[p1] - c;
    D2H(ctx, results, ws.d_results, sizeof(PlPoseResult), p0, p1 - p0, s);
    D2H(ctx, m12_pt, ws.d_m12p, 4, a, an, s);
    D2H(ctx, m12_ls, ws.d_m12l, 4, c, cn, s);
    D2H(ctx, inl_pt, ws.d_inlp, 1, a, an, s);
    D2H(ctx, inl_ls, ws.d_inll, 1, c, cn, s);
    return 0;
}

// Pipeline chunking of the host-buffer entry point: small first chunks (the GPU starts working after a few MB have
// crossed PCIe), then chunks of about two thirds of the SM count in pairs (K2 runs one pair per SM; the rest of the
// chip keeps running the next chunk's distance tiles on the other compute stream).
// With batches in flight behind one another (plstvo_track_batch_async) the previous batch's kernels already hide the copy:
// no ramp, the resident pass's chunking (two launches per pass) is used instead.
std::vector<int> chunk_schedule(int B, int sm_count, bool pipelined) {
    static const int forced = getenv("PLSTVO_E2E_CHUNK") ? atoi(getenv("PLSTVO_E2E_CHUNK")) : 0;
    std::vector<int> bounds{0};
    if (forced > 0 || pipelined) {
        const int step = forced > 0 ? forced : std::max(1, std::max(std::min(B, sm_count), (B + 1) / 2));
        for (int p = step; p < B; p += step) bounds.push_back(p);
        bounds.push_back(B);
        return bounds;
    }
    const char* list = getenv("PLSTVO_E2E_BOUNDS");         // tuning knob: explicit chunk ends, e.g. "74,293"
    if (list && *list) {
        for (const char* c = list; *c;) {
            const int v = atoi(c);
            if (v > bounds.back() && v < B) bounds.push_back(v);
            while (*c && *c != ',') ++c;
            if (*c == ',') ++c;
        }
        bounds.push_back(B);
        return bounds;
    }
    // ramp 1/6, 1/3, 2/3 of the SM count, then equal chunks of at most one pair per SM
    int p = 0;
    for (int c = std::max(8, sm_count / 6); c < sm_count && p + c < B; c *= 2) {
        p += c;
        bounds.push_back(p);
    }
    const int rest = B - p;
    if (rest > 0) {
        const int n = (rest + sm_count - 1) / sm_count;
        for (int k = 1; k <= n; ++k) bounds.push_back(p + (int)((long)rest * k / n));
    }
    return bounds;
}

int run_chunk(const Workspace& ws, int sm_count) {
    static const int forced = getenv("PLSTVO_RUN_CHUNK") ? atoi(getenv("PLSTVO_RUN_CHUNK")) : 0;
    if (forced > 0) return forced;
    return std::max(1, std::max(std::min(ws.B, sm_count), (ws.B + 1) / 2));   // two launches per pass (measured best)
}

// resident pass: K1 / K2 over the whole batch, chunked over two streams so that the (latency-bound) per-pair
// solver of chunk i overlaps the (throughput-bound) distance tiles of chunk i+1
int ws_run(PlContext* ctx, Workspace& ws, bool have_level) {
    if (ws.B == 0) return 0;
    const int chunk = run_chunk(ws, ctx->sm_count);
    cudaEvent_t start = next_event(ctx);
    CK(ctx, cudaEventRecord(start, ctx->s_main));
    CK(ctx, cudaStreamWaitEvent(ctx->s_alt, start, 0));
    int k = 0;
    for (int p0 = 0; p0 < ws.B; p0 += chunk, ++k) {
        const int p1 = std::min(ws.B, p0 + chunk);
        cudaStream_t s = (k & 1) ? ctx->s_alt : ctx->s_main;
        int rc = ws_launch_match(ctx, ws, p0, p1, s);
        if (rc) return rc;
        rc = ws_launch_solve(ctx, ws, p0, p1, have_level, s);
        if (rc) return rc;
    }
    cudaEvent_t done = next_event(ctx);
    CK(ctx, cudaEventRecord(done, ctx->s_alt));
    CK(ctx, cudaStreamWaitEvent(ctx->s_main, done, 0));
    return 0;
}

}  // namespace

// =====================================================================================================
extern "C" {

int plstvo_version(void) { return PLSTVO_VERSION; }

int plstvo_create(int device, PlContext** out) {
    if (!out) return PLSTVO_E_INVALID;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) return PLSTVO_E_NO_DEVICE;
    if (device < 0) {
        if (cudaGetDevice(&device) != cudaSuccess) return PLSTVO_E_NO_DEVICE;
    }
    if (device >= n) return PLSTVO_E_NO_DEVICE;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return PLSTVO_E_NO_DEVICE;
    if (prop.major != 10) return PLSTVO_E_NO_DEVICE;   // the kernels are built for sm_100a only
    if (cudaSetDevice(device) != cudaSuccess) return PLSTVO_E_NO_DEVICE;
    PlContext* ctx = new PlContext();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    cudaStreamCreateWithFlags(&ctx->s_main, cudaStreamNonBlocking);
    cudaStreamCreateWithFlags(&ctx->s_alt, cudaStreamNonBlocking);
    cudaStreamCreateWithFlags(&ctx->s_h2d, cudaStreamNonBlocking);
    cudaStreamCreateWithFlags(&ctx->s_d2h, cudaStreamNonBlocking);
    *out = ctx;
    return 0;
}

void plstvo_destroy(PlContext* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    ctx->ws.release();
    ctx->ws_async[0].release();
    ctx->ws_async[1].release();
    for (auto& e : ctx->slot_done)
        if (e) cudaEventDestroy(e);
    ctx->scratch.release();
    for (auto& b : ctx->gn_in) b.release();
    for (auto& b : ctx->gn_out) b.release();
    ctx->arena_grid.release(); ctx->arena_lift_pt.release(); ctx->arena_lift_ls.release();
    ctx->arena_stereo.release();
    for (auto& b : ctx->arena_track_stereo) b.release();
    for (auto& b : ctx->gs_in) b.release();
    ctx->gs_rec_pt.release(); ctx->gs_rec_ls.release();
    for (cudaEvent_t e : ctx->events) cudaEventDestroy(e);
    for (void* h : ctx->h_staging)
        if (h) cudaFreeHost(h);
    cudaStreamDestroy(ctx->s_main);
    cudaStreamDestroy(ctx->s_alt);
    cudaStreamDestroy(ctx->s_h2d);
    cudaStreamDestroy(ctx->s_d2h);
    delete ctx;
}

const char* plstvo_last_error(const PlContext* ctx) { return ctx ? ctx->err.c_str() : "no context"; }

void plstvo_default_config(PlConfig* c) {   // src/config.cpp:36-113
    c->has_points = 1; c->has_lines = 1; c->best_lr_matches = 1; c->use_motion_model = 0;
    c->min_features = 10; c->max_iters = 5; c->max_iters_ref = 10; c->solver_mode = 0;
    c->min_ratio_12_p = 0.9; c->min_ratio_12_l = 0.9; c->homog_th = 1e-7; c->min_error = 1e-7;
    c->min_error_change = 1e-7; c->inlier_k = 4.0; c->lsd_scale = 1.2;
}

void plstvo_kitti_config(PlConfig* c) {   // config/config/config_kitti.yaml:19,27,45
    plstvo_default_config(c);
    c->min_ratio_12_p = 0.75;
    c->min_ratio_12_l = 0.75;
    c->inlier_k = 1.2;
}

int plstvo_synchronize(PlContext* ctx) {
    if (!ctx) return PLSTVO_E_INVALID;
    LOCK(ctx);
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaStreamSynchronize(ctx->s_h2d));
    CK(ctx, cudaStreamSynchronize(ctx->s_main));
    CK(ctx, cudaStreamSynchronize(ctx->s_alt));
    CK(ctx, cudaStreamSynchronize(ctx->s_d2h));
    return 0;
}

void* plstvo_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) return nullptr;
    return p;
}
void plstvo_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

int64_t plstvo_launch_count(const PlContext* ctx) { return ctx ? ctx->launches : 0; }

// ---- matching.h surface -------------------------------------------------------------------------------
int plstvo_match_batch(PlContext* ctx, int B, const uint8_t* d1, const int32_t* off1, const uint8_t* d2,
                       const int32_t* off2, float nnr, int best_lr_matches, int32_t* m12, int32_t* counts) {
    if (!ctx) return PLSTVO_E_INVALID;
    LOCK(ctx);
    if (B < 0 || (B > 0 && (!off1 || !off2 || !m12))) return fail(ctx, PLSTVO_E_INVALID, "bad arguments");
    if (B == 0) return 0;
    CK(ctx, cudaSetDevice(ctx->device));
    // express the problems as a points-only frame batch
    std::vector<int32_t> zeros((size_t)B + 1, 0);
    PlFrameBatch a{}, b{};
    a.B = b.B = B;
    a.pt_off = off1; b.pt_off = off2;
    a.ls_off = b.ls_off = zeros.data();
    a.pdesc = d1; b.pdesc = d2;
    int rc = validate_frames(ctx, &a, &b, false);
    if (rc) return rc;
    PlConfig cfg;
    plstvo_default_config(&cfg);
    cfg.has_lines = 0;
    cfg.best_lr_matches = best_lr_matches;
    Workspace& ws = ctx->ws;
    rc = ws_prepare(ctx, ws, nullptr, &cfg, &a, &b, false, false);
    if (rc) return rc;
    ws.planned = false;                          // this entry point patches the plan below: never reuse it
    for (auto& pr : ws.problems) pr.nnr = nnr;   // the caller's float, not the config's double
    CK(ctx, cudaMemcpyAsync(ws.d_problems.p, ws.problems.data(), ws.problems.size() * sizeof(MatchProblem),
                            cudaMemcpyHostToDevice, ctx->s_h2d));
    rc = ws_upload_range(ctx, ws, &a, &b, nullptr, 0, B, false, ctx->s_h2d);
    if (rc) return rc;
    cudaEvent_t up = next_event(ctx);
    CK(ctx, cudaEventRecord(up, ctx->s_h2d));
    CK(ctx, cudaStreamWaitEvent(ctx->s_main, up, 0));
    rc = ws_launch_match(ctx, ws, 0, B, ctx->s_main);
    if (rc) return rc;
    // finalize only the point problems (even indices): compact view
    CK(ctx, ctx->scratch.ensure((size_t)B * (sizeof(MatchProblem) + 4)));
    std::vector<MatchProblem> pts((size_t)B);
    for (int p = 0; p < B; ++p) pts[p] = ws.problems[(size_t)2 * p];
    MatchProblem* d_pts = ctx->scratch.as<MatchProblem>();
    int32_t* d_counts = reinterpret_cast<int32_t*>(d_pts + B);
    CK(ctx, cudaMemcpyAsync(d_pts, pts.data(), (size_t)B * sizeof(MatchProblem), cudaMemcpyHostToDevice, ctx->s_main));
    CK(ctx, launch_match_finalize(d_pts, B, ws.max_n2, d_counts, ctx->s_main));
    ctx->launches++;
    CK(ctx, cudaMemcpyAsync(m12, ws.d_m12p.p, (size_t)off1[B] * 4, cudaMemcpyDeviceToHost, ctx->s_main));
    std::vector<int32_t> cnt((size_t)B);
    CK(ctx, cudaMemcpyAsync(cnt.data(), d_counts, (size_t)B * 4, cudaMemcpyDeviceToHost, ctx->s_main));
    CK(ctx, cudaStreamSynchronize(ctx->s_main));
    long total = 0;
    for (int p = 0; p < B; ++p) {
        if (counts) counts[p] = cnt[p];
        total += cnt[p];
    }
    return (int)total;
}

int plstvo_match(PlContext* ctx, const uint8_t* d1, int n1, const uint8_t* d2, int n2, int stride_bytes,
                 float nnr, int best_lr_matches, int32_t* m12) {
    if (!ctx) return PLSTVO_E_INVALID;
    LOCK(ctx);
    if (stride_bytes != PLSTVO_DESC_BYTES) return fail(ctx, PLSTVO_E_INVALID, "descriptor rows must be 32 contiguous bytes");
    if (n1 < 0 || n2 < 0) return fail(ctx, PLSTVO_E_INVALID, "negative row count");
    if (n1 == 0) return 0;
    if (!m12) return fail(ctx, PLSTVO_E_INVALID, "null output");
    const int32_t o1[2] = {0, n1}, o2[2] = {0, n2};
    return plstvo_match_batch(ctx, 1, d1, o1, d2, o2, nnr, best_lr_matches, m12, nullptr);
}

int plstvo_match_nnr(PlContext* ctx, const uint8_t* d1, int n1, const uint8_t* d2, int n2, int stride_bytes,
                     float nnr, int32_t* m12) {
    return plstvo_match(ctx, d1, n1, d2, n2, stride_bytes, nnr, 0, m12);
}

// ---- matchGrid (stereo step) -------------------------------------------------------------------------------------
static int match_grid_common(PlContext* ctx, bool lines, int B, int rows, int cols, PlGridWindow w, int best_lr,
                             double ratio, double line_sim_th, const int32_t* q_off, const int32_t* q_cell,
                             const uint8_t* d1, const int32_t* t_off, const int32_t* t_cell, const double* t_line,
                             const double* t_dir, const uint8_t* d2, int32_t* m12, int32_t* counts) {
    if (!ctx) return PLSTVO_E_INVALID;
    LOCK(ctx);
    if (B < 0 || rows <= 0 || cols <= 0 || rows * cols > 8192) return fail(ctx, PLSTVO_E_INVALID, "bad grid");
    if (B == 0) return 0;
    if (!q_off || !t_off || !m12 || q_off[0] || t_off[0]) return fail(ctx, PLSTVO_E_INVALID, "bad offsets");
    CK(ctx, cudaSetDevice(ctx->device));
    constexpr int CAP = 128;                      // candidates per query window (the reference has no limit; typical: ~10)
    const int qw = lines ? 4 : 2;
    const size_t N1 = q_off[B], N2 = t_off[B];
    for (int p = 0; p < B; ++p) {
        const int n1 = q_off[p + 1] - q_off[p], n2 = t_off[p + 1] - t_off[p];
        if (n1 < 0 || n2 < 0) return fail(ctx, PLSTVO_E_INVALID, "offsets are not non-decreasing");
        if (n1 > PLSTVO_MAX_FEATURES || n2 > PLSTVO_MAX_FEATURES) return fail(ctx, PLSTVO_E_TOO_LARGE, "more than 65535 features");
    }
    if ((N1 && (!q_cell || !d1)) || (N2 && (!d2 || (lines ? (!t_line || !t_dir) : !t_cell))))
        return fail(ctx, PLSTVO_E_INVALID, "null input array");
    const size_t per_train_cells = lines ? (size_t)std::max(rows, cols) + 2 : 1;
    // one arena for inputs, outputs and scratch
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const size_t o_qcell = take(N1 * qw * 4), o_d1 = take(N1 * 32), o_d2 = take(N2 * 32);
    const size_t o_tcell = take(lines ? 0 : N2 * 8), o_tline = take(lines ? N2 * 32 : 0), o_tdir = take(lines ? N2 * 16 : 0);
    const size_t o_m12 = take(N1 * 4), o_cnt = take((size_t)B * 4), o_items = take(N2 * per_train_cells * 4);
    const size_t o_qpairs = take(N1 * CAP * 8), o_qcount = take(N1 * 4), o_tcount = take(N2 * 4);
    const size_t o_tstart = take((N2 + B) * 4), o_tslots = take(N1 * CAP * 4), o_seen = take(N1 * CAP), o_m21 = take(N2 * 4);
    const size_t o_prob = take((size_t)B * sizeof(GridProblem));
    DevBuf& arena = ctx->arena_grid;
    CK(ctx, arena.ensure(off));
    uint8_t* base = arena.as<uint8_t>();
    std::vector<GridProblem> probs((size_t)B);
    for (int p = 0; p < B; ++p) {
        GridProblem& g = probs[p];
        const size_t a = q_off[p], b = t_off[p];
        g.n1 = q_off[p + 1] - q_off[p];
        g.n2 = t_off[p + 1] - t_off[p];
        g.q_cell = reinterpret_cast<int32_t*>(base + o_qcell) + a * qw;
        g.d1 = base + o_d1 + a * 32;
        g.t_cell = lines ? nullptr : reinterpret_cast<int32_t*>(base + o_tcell) + b * 2;
        g.t_line = lines ? reinterpret_cast<double*>(base + o_tline) + b * 4 : nullptr;
        g.t_dir = lines ? reinterpret_cast<double*>(base + o_tdir) + b * 2 : nullptr;
        g.d2 = base + o_d2 + b * 32;
        g.m12 = reinterpret_cast<int32_t*>(base + o_m12) + a;
        g.count = reinterpret_cast<int32_t*>(base + o_cnt) + p;
        g.grid_items = reinterpret_cast<int32_t*>(base + o_items) + b * per_train_cells;
        g.q_pairs = reinterpret_cast<int2*>(base + o_qpairs) + a * CAP;
        g.q_count = reinterpret_cast<int32_t*>(base + o_qcount) + a;
        g.t_count = reinterpret_cast<int32_t*>(base + o_tcount) + b;
        g.t_start = reinterpret_cast<int32_t*>(base + o_tstart) + b + p;
        g.t_slots = reinterpret_cast<int32_t*>(base + o_tslots) + a * CAP;
        g.seen = base + o_seen + a * CAP;
        g.m21 = reinterpret_cast<int32_t*>(base + o_m21) + b;
    }
    cudaStream_t s = ctx->s_main;
    auto up = [&](size_t o, const void* src, size_t bytes) -> cudaError_t {
        return (src && bytes) ? cudaMemcpyAsync(base + o, src, bytes, cudaMemcpyHostToDevice, s) : cudaSuccess;
    };
    CK(ctx, up(o_qcell, q_cell, N1 * qw * 4));
    CK(ctx, up(o_d1, d1, N1 * 32));
    CK(ctx, up(o_d2, d2, N2 * 32));
    if (lines) {
        CK(ctx, up(o_tline, t_line, N2 * 32));
        CK(ctx, up(o_tdir, t_dir, N2 * 16));
    } else {
        CK(ctx, up(o_tcell, t_cell, N2 * 8));
    }
    CK(ctx, up(o_prob, probs.data(), (size_t)B * sizeof(GridProblem)));
    GridParams prm{rows, cols, CAP, best_lr ? 1 : 0, w, ratio, line_sim_th};
    CK(ctx, launch_match_grid(reinterpret_cast<GridProblem*>(base + o_prob), B, prm, lines, s));
    ctx->launches++;
    std::vector<int32_t> cnt((size_t)B);
    if (N1) CK(ctx, cudaMemcpyAsync(m12, base + o_m12, N1 * 4, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaMemcpyAsync(cnt.data(), base + o_cnt, (size_t)B * 4, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    long total = 0;
    for (int p = 0; p < B; ++p) {
        if (cnt[p] < 0) return fail(ctx, cnt[p], "matchGrid: more than 128 candidates in one query window");
        if (counts) counts[p] = cnt[p];
        total += cnt[p];
    }
    return (int)total;
}

int plstvo_match_grid_points(PlContext* ctx, int B, int grid_rows, int grid_cols, PlGridWindow w, int best_lr_matches,
                             double min_ratio_12_p, const int32_t* q_off, const int32_t* q_cell, const uint8_t* d1,
                             const int32_t* t_off, const int32_t* t_cell, const uint8_t* d2, int32_t* m12,
                             int32_t* counts) {
    return match_grid_common(ctx, false, B, grid_rows, grid_cols, w, best_lr_matches, min_ratio_12_p, 0.0, q_off, q_cell, d1,
                             t_off, t_cell, nullptr, nullptr, d2, m12, counts);
}

int plstvo_match_grid_lines(PlContext* ctx, int B, int grid_rows, int grid_cols, PlGridWindow w, int best_lr_matches,
                            double min_ratio_12_p, double line_sim_th, const int32_t* q_off, const int32_t* q_line,
                            const uint8_t* d1, const int32_t* t_off, const double* t_line, const double* t_dir,
                            const uint8_t* d2, int32_t* m12, int32_t* counts) {
    return match_grid_common(ctx, true, B, grid_rows, grid_cols, w, best_lr_matches, min_ratio_12_p, line_sim_th, q_off,
                             q_line, d1, t_off, nullptr, t_line, t_dir, d2, m12, counts);
}

// ---- 3-D lifting of the stereo matches (src/stereoFrame.cpp:149-172, :348-397) ------------------------------
void plstvo_default_stereo_config(PlStereoConfig* c) {   // src/config.cpp:58-69, :96, :106
    if (!c) return;
    c->max_dist_epip = 1.0; c->min_disp = 1.0; c->ls_min_disp_ratio = 0.7; c->line_horiz_th = 0.1;
    c->stereo_overlap_th = 0.75; c->orb_scale_factor = 1.2; c->lsd_scale = 1.2;
}

namespace {
struct LiftArena {
    size_t off = 0;
    size_t take(size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; }
};
int lift_check_offsets(PlContext* ctx, int B, const int32_t* l_off, const int32_t* r_off) {
    if (!l_off || !r_off || l_off[0] || r_off[0]) return fail(ctx, PLSTVO_E_INVALID, "bad offsets");
    for (int p = 0; p < B; ++p) {
        const int n1 = l_off[p + 1] - l_off[p], n2 = r_off[p + 1] - r_off[p];
        if (n1 < 0 || n2 < 0) return fail(ctx, PLSTVO_E_INVALID, "offsets are not non-decreasing");
        if (n1 > PLSTVO_MAX_FEATURES || n2 > PLSTVO_MAX_FEATURES) return fail(ctx, PLSTVO_E_TOO_LARGE, "more than 65535 features");
    }
    return 0;
}
}  // namespace

int plstvo_stereo_lift_points(PlContext* ctx, const PlCamera* cam, const PlStereoConfig* scfg, int B, const int32_t* l_off,
                              const float* kp_l, const int32_t* octave_l, const uint8_t* desc_l, const int32_t* r_off,
                              const float* kp_r, const int32_t* m12, double* pt_pl, double* pt_disp, double* pt_P,
                              double* pt_sigma2, int32_t* pt_level, uint8_t* pdesc_out, int32_t* src_idx, int32_t* counts) {
    if (!ctx) return PLSTVO_E_INVALID;
    LOCK(ctx);
    if (!cam || !scfg || B < 0) return fail(ctx, PLSTVO_E_INVALID, "null camera / config or negative batch size");
    if (B == 0) return 0;
    int rc = lift_check_offsets(ctx, B, l_off, r_off);
    if (rc) return rc;
    const size_t N1 = l_off[B], N2 = r_off[B];
    if (N1 && (!kp_l || !octave_l || !desc_l || !m12)) return fail(ctx, PLSTVO_E_INVALID, "null input array");
    if (N2 && !kp_r) return fail(ctx, PLSTVO_E_INVALID, "null input array");
    CK(ctx, cudaSetDevice(ctx->device));
    LiftArena a;
    const size_t o_loff = a.take((size_t)(B + 1) * 4), o_roff = a.take((size_t)(B + 1) * 4), o_kpl = a.take(N1 * 8);
    const size_t o_oct = a.take(N1 * 4), o_desc = a.take(N1 * 32), o_kpr = a.take(N2 * 8), o_m12 = a.take(N1 * 4);
    const size_t o_pl = a.take(N1 * 16), o_disp = a.take(N1 * 8), o_P = a.take(N1 * 24), o_s2 = a.take(N1 * 8);
    const size_t o_lvl = a.take(N1 * 4), o_dout = a.take(N1 * 32), o_src = a.take(N1 * 4), o_cnt = a.take((size_t)B * 4);
    DevBuf& arena = ctx->arena_lift_pt;
    CK(ctx, arena.ensure(a.off));
    uint8_t* base = arena.as<uint8_t>();
    cudaStream_t s = ctx->s_main;
    auto up = [&](size_t o, const void* src, size_t bytes) -> cudaError_t {
        return (src && bytes) ? cudaMemcpyAsync(base + o, src, bytes, cudaMemcpyHostToDevice, s) : cudaSuccess;
    };
    auto down = [&](void* dst, size_t o, size_t bytes) -> cudaError_t {
        return (dst && bytes) ? cudaMemcpyAsync(dst, base + o, bytes, cudaMemcpyDeviceToHost, s) : cudaSuccess;
    };
    CK(ctx, up(o_loff, l_off, (size_t)(B + 1) * 4));
    CK(ctx, up(o_roff, r_off, (size_t)(B + 1) * 4));
    CK(ctx, up(o_kpl, kp_l, N1 * 8));
    CK(ctx, up(o_oct, octave_l, N1 * 4));
    CK(ctx, up(o_desc, desc_l, N1 * 32));
    CK(ctx, up(o_kpr, kp_r, N2 * 8));
    CK(ctx, up(o_m12, m12, N1 * 4));
    auto I = [&](size_t o) { return reinterpret_cast<int32_t*>(base + o); };
    auto D = [&](size_t o) { return reinterpret_cast<double*>(base + o); };
    auto F = [&](size_t o) { return reinterpret_cast<float*>(base + o); };
    CK(ctx, launch_lift_points(*cam, *scfg, B, I(o_loff), F(o_kpl), I(o_oct), base + o_desc, I(o_roff), F(o_kpr), I(o_m12),
                               D(o_pl), D(o_disp), D(o_P), D(o_s2), I(o_lvl), base + o_dout, I(o_src), I(o_cnt), s));
    ctx->launches++;
    std::vector<int32_t> cnt((size_t)B);
    CK(ctx, down(pt_pl, o_pl, N1 * 16));
    CK(ctx, down(pt_disp, o_disp, N1 * 8));
    CK(ctx, down(pt_P, o_P, N1 * 24));
    CK(ctx, down(pt_sigma2, o_s2, N1 * 8));
    CK(ctx, down(pt_level, o_lvl, N1 * 4));
    CK(ctx, down(pdesc_out, o_dout, N1 * 32));
    CK(ctx, down(src_idx, o_src, N1 * 4));
    CK(ctx, down(cnt.data(), o_cnt, (size_t)B * 4));
    CK(ctx, cudaStreamSynchronize(s));
    long total = 0;
    for (int p = 0; p < B; ++p) {
        if (counts) counts[p] = cnt[p];
        total += cnt[p];
    }
    return (int)total;
}

int plstvo_stereo_lift_lines(PlContext* ctx, const PlCamera* cam, const PlStereoConfig* scfg, int B, const int32_t* l_off,
                             const float* seg_l, const float* angle_l, const int32_t* octave_l, const uint8_t* desc_l,
                             const int32_t* r_off, const float* seg_r, const int32_t* m12, double* ls_spl, double* ls_epl,
                             double* ls_sdisp, double* ls_edisp, double* ls_sP, double* ls_eP, double* ls_le,
                             double* ls_angle, double* ls_sigma2, int32_t* ls_level, uint8_t* ldesc_out, int32_t* src_idx,
                             int32_t* counts) {
    if (!ctx) return PLSTVO_E_INVALID;
    LOCK(ctx);
    if (!cam || !scfg || B < 0) return fail(ctx, PLSTVO_E_INVALID, "null camera / config or negative batch size");
    if (B == 0) return 0;
    int rc = lift_check_offsets(ctx, B, l_off, r_off);
    if (rc) return rc;
    const size_t N1 = l_off[B], N2 = r_off[B];
    if (N1 && (!seg_l || !angle_l || !octave_l || !desc_l || !m12)) return fail(ctx, PLSTVO_E_INVALID, "null input array");
    if (N2 && !seg_r) return fail(ctx, PLSTVO_E_INVALID, "null input array");
    CK(ctx, cudaSetDevice(ctx->device));
    LiftArena a;
    const size_t o_loff = a.take((size_t)(B + 1) * 4), o_roff = a.take((size_t)(B + 1) * 4), o_segl = a.take(N1 * 16);
    const size_t o_ang = a.take(N1 * 4), o_oct = a.take(N1 * 4), o_desc = a.take(N1 * 32), o_segr = a.take(N2 * 16);
    const size_t o_m12 = a.take(N1 * 4), o_spl = a.take(N1 * 16), o_epl = a.take(N1 * 16), o_sd = a.take(N1 * 8);
    const size_t o_ed = a.take(N1 * 8), o_sP = a.take(N1 * 24), o_eP = a.take(N1 * 24), o_le = a.take(N1 * 24);
    const size_t o_angd = a.take(N1 * 8), o_s2 = a.take(N1 * 8), o_lvl = a.take(N1 * 4), o_dout = a.take(N1 * 32);
    const size_t o_src = a.take(N1 * 4), o_cnt = a.take((size_t)B * 4);
    DevBuf& arena = ctx->arena_lift_ls;
    CK(ctx, arena.ensure(a.off));
    uint8_t* base = arena.as<uint8_t>();
    cudaStream_t s = ctx->s_main;
    auto up = [&](size_t o, const void* src, size_t bytes) -> cudaError_t {
        return (src && bytes) ? cudaMemcpyAsync(base + o, src, bytes, cudaMemcpyHostToDevice, s) : cudaSuccess;
    };
    auto down = [&](void* dst, size_t o, size_t bytes) -> cudaError_t {
        return (dst && bytes) ? cudaMemcpyAsync(dst, base + o, bytes, cudaMemcpyDeviceToHost, s) : cudaSuccess;
    };
    CK(ctx, up(o_loff, l_off, (size_t)(B + 1) * 4));
    CK(ctx, up(o_roff, r_off, (size_t)(B + 1) * 4));
    CK(ctx, up(o_segl, seg_l, N1 * 16));
    CK(ctx, up(o_ang, angle_l, N1 * 4));
    CK(ctx, up(o_oct, octave_l, N1 * 4));
    CK(ctx, up(o_desc, desc_l, N1 * 32));
    CK(ctx, up(o_segr, seg_r, N2 * 16));
    CK(ctx, up(o_m12, m12, N1 * 4));
    auto I = [&](size_t o) { return reinterpret_cast<int32_t*>(base + o); };
    auto D = [&](size_t o) { return reinterpret_cast<double*>(base + o); };
    auto F = [&](size_t o) { return reinterpret_cast<float*>(base + o); };
    CK(ctx, launch_lift_lines(*cam, *scfg, B, I(o_loff), F(o_segl), F(o_ang), I(o_oct), base + o_desc, I(o_roff), F(o_segr),
                              I(o_m12), D(o_spl), D(o_epl), D(o_sd), D(o_ed), D(o_sP), D(o_eP), D(o_le), D(o_angd), D(o_s2),
                              I(o_lvl), base + o_dout, I(o_src), I(o_cnt), s));
    ctx->launches++;
    std::vector<int32_t> cnt((size_t)B);
    CK(ctx, down(ls_spl, o_spl, N1 * 16));
    CK(ctx, down(ls_epl, o_epl, N1 * 16));
    CK(ctx, down(ls_sdisp, o_sd, N1 * 8));
    CK(ctx, down(ls_edisp, o_ed, N1 * 8));
    CK(ctx, down(ls_sP, o_sP, N1 * 24));
    CK(ctx, down(ls_eP, o_eP, N1 * 24));
    CK(ctx, down(ls_le, o_le, N1 * 24));
    CK(ctx, down(ls_angle, o_angd, N1 * 8));
    CK(ctx, down(ls_sigma2, o_s2, N1 * 8));
    CK(ctx, down(ls_level, o_lvl, N1 * 4));
    CK(ctx, down(ldesc_out, o_dout, N1 * 32));
    CK(ctx, down(src_idx, o_src, N1 * 4));
    CK(ctx, down(cnt.data(), o_cnt, (size_t)B * 4));
    CK(ctx, cudaStreamSynchronize(s));
    long total = 0;
    for (int p = 0; p < B; ++p) {
        if (counts) counts[p] = cnt[p];
        total += cnt[p];
    }
    return (int)total;
}

// ---- matchStereoPoints / matchStereoLines in one device pass (src/stereoFrame.cpp:120-173, :309-398) ----------------
void plstvo_default_stereo_match_config(PlStereoMatchConfig* c) {   // include/stereoFrame.h:51-52, src/config.cpp:51, :60, :63, :91
    if (!c) return;
    c->grid_rows = 48; c->grid_cols = 64; c->matching_s_ws = 10; c->best_lr_matches = 1;
    c->min_ratio_12_p = 0.9; c->line_sim_th = 0.75;
}

namespace {
struct StereoOut {   // host destinations of the lifted records (points use the first seven)
    int32_t* m12; double *a_pl, *a_disp, *a_P, *a_s2; int32_t* level; uint8_t* desc; int32_t *src, *counts;
    double *epl, *edisp, *eP, *le, *angle;   // lines only
};

int match_stereo_common(PlContext* ctx, bool lines, const PlCamera* cam, const PlStereoMatchConfig* mc, const PlStereoConfig* sc,
                        int B, const int32_t* l_off, const float* xy_l, const float* angle_l, const int32_t* octave_l,
                        const uint8_t* desc_l, const int32_t* r_off, const float* xy_r, const uint8_t* desc_r,
                        const StereoOut& out) {
    if (!ctx) return PLSTVO_E_INVALID;
    LOCK(ctx);
    if (!cam || !mc || !sc || B < 0) return fail(ctx, PLSTVO_E_INVALID, "null camera / config or negative batch size");
    const int rows = mc->grid_rows, cols = mc->grid_cols;
    if (rows <= 0 || cols <= 0 || rows * cols > 8192 || cam->width <= 0 || cam->height <= 0)
        return fail(ctx, PLSTVO_E_INVALID, "bad grid or image size");
    if (B == 0) return 0;
    int rc = lift_check_offsets(ctx, B, l_off, r_off);
    if (rc) return rc;
    const size_t N1 = l_off[B], N2 = r_off[B];
    if (N1 && (!xy_l || !octave_l || !desc_l || (lines && !angle_l))) return fail(ctx, PLSTVO_E_INVALID, "null input array");
    if (N2 && (!xy_r || !desc_r)) return fail(ctx, PLSTVO_E_INVALID, "null input array");
    CK(ctx, cudaSetDevice(ctx->device));
    constexpr int CAP = 128;
    const int cw = lines ? 4 : 2;                 // floats per feature (segment / key point) and ints per query cell record
    const size_t per_train_cells = lines ? (size_t)std::max(rows, cols) + 2 : 1;
    LiftArena a;
    // raw inputs
    const size_t o_loff = a.take((size_t)(B + 1) * 4), o_roff = a.take((size_t)(B + 1) * 4), o_xyl = a.take(N1 * cw * 4);
    const size_t o_xyr = a.take(N2 * cw * 4), o_ang = a.take(lines ? N1 * 4 : 0), o_oct = a.take(N1 * 4);
    const size_t o_d1 = a.take(N1 * 32), o_d2 = a.take(N2 * 32);
    // matchGrid
    const size_t o_qcell = a.take(N1 * cw * 4), o_tcell = a.take(lines ? 0 : N2 * 8), o_tline = a.take(lines ? N2 * 32 : 0);
    const size_t o_tdir = a.take(lines ? N2 * 16 : 0), o_m12 = a.take(N1 * 4), o_gcnt = a.take((size_t)B * 4);
    const size_t o_items = a.take(N2 * per_train_cells * 4), o_qpairs = a.take(N1 * CAP * 8), o_qcount = a.take(N1 * 4);
    const size_t o_tcount = a.take(N2 * 4), o_tstart = a.take((N2 + B) * 4), o_tslots = a.take(N1 * CAP * 4);
    const size_t o_seen = a.take(N1 * CAP), o_m21 = a.take(N2 * 4), o_prob = a.take((size_t)B * sizeof(GridProblem));
    // lifted records
    const size_t o_pl = a.take(N1 * 16), o_disp = a.take(N1 * 8), o_P = a.take(N1 * 24), o_s2 = a.take(N1 * 8);
    const size_t o_lvl = a.take(N1 * 4), o_dout = a.take(N1 * 32), o_src = a.take(N1 * 4), o_cnt = a.take((size_t)B * 4);
    const size_t o_epl = a.take(lines ? N1 * 16 : 0), o_edisp = a.take(lines ? N1 * 8 : 0), o_eP = a.take(lines ? N1 * 24 : 0);
    const size_t o_le = a.take(lines ? N1 * 24 : 0), o_angd = a.take(lines ? N1 * 8 : 0);
    DevBuf& arena = ctx->arena_stereo;
    CK(ctx, arena.ensure(a.off));
    uint8_t* base = arena.as<uint8_t>();
    auto I = [&](size_t o) { return reinterpret_cast<int32_t*>(base + o); };
    auto D = [&](size_t o) { return reinterpret_cast<double*>(base + o); };
    auto F = [&](size_t o) { return reinterpret_cast<float*>(base + o); };
    std::vector<GridProblem> probs((size_t)B);
    for (int p = 0; p < B; ++p) {
        GridProblem& g = probs[p];
        const size_t qa = l_off[p], tb = r_off[p];
        g.n1 = l_off[p + 1] - l_off[p];
        g.n2 = r_off[p + 1] - r_off[p];
        g.q_cell = I(o_qcell) + qa * cw;
        g.d1 = base + o_d1 + qa * 32;
        g.t_cell = lines ? nullptr : I(o_tcell) + tb * 2;
        g.t_line = lines ? D(o_tline) + tb * 4 : nullptr;
        g.t_dir = lines ? D(o_tdir) + tb * 2 : nullptr;
        g.d2 = base + o_d2 + tb * 32;
        g.m12 = I(o_m12) + qa;
        g.count = I(o_gcnt) + p;
        g.grid_items = I(o_items) + tb * per_train_cells;
        g.q_pairs = reinterpret_cast<int2*>(base + o_qpairs) + qa * CAP;
        g.q_count = I(o_qcount) + qa;
        g.t_count = I(o_tcount) + tb;
        g.t_start = I(o_tstart) + tb + p;
        g.t_slots = I(o_tslots) + qa * CAP;
        g.seen = base + o_seen + qa * CAP;
        g.m21 = I(o_m21) + tb;
    }
    cudaStream_t s = ctx->s_main;
    auto up = [&](size_t o, const void* src, size_t bytes) -> cudaError_t {
        return (src && bytes) ? cudaMemcpyAsync(base + o, src, bytes, cudaMemcpyHostToDevice, s) : cudaSuccess;
    };
    auto down = [&](void* dst, size_t o, size_t bytes) -> cudaError_t {
        return (dst && bytes) ? cudaMemcpyAsync(dst, base + o, bytes, cudaMemcpyDeviceToHost, s) : cudaSuccess;
    };
    CK(ctx, up(o_loff, l_off, (size_t)(B + 1) * 4));
    CK(ctx, up(o_roff, r_off, (size_t)(B + 1) * 4));
    CK(ctx, up(o_xyl, xy_l, N1 * cw * 4));
    CK(ctx, up(o_xyr, xy_r, N2 * cw * 4));
    if (lines) CK(ctx, up(o_ang, angle_l, N1 * 4));
    CK(ctx, up(o_oct, octave_l, N1 * 4));
    CK(ctx, up(o_d1, desc_l, N1 * 32));
    CK(ctx, up(o_d2, desc_r, N2 * 32));
    CK(ctx, up(o_prob, probs.data(), (size_t)B * sizeof(GridProblem)));
    // 1. grid coordinates (:47-48: inv_width = GRID_COLS / image width, inv_height = GRID_ROWS / image height)
    const double inv_w = cols / static_cast<double>(cam->width), inv_h = rows / static_cast<double>(cam->height);
    if (lines)
        CK(ctx, launch_stereo_cells_lines((int)N1, (int)N2, inv_w, inv_h, F(o_xyl), F(o_xyr), I(o_qcell), D(o_tline), D(o_tdir), s));
    else
        CK(ctx, launch_stereo_cells_points((int)N1, (int)N2, inv_w, inv_h, F(o_xyl), F(o_xyr), I(o_qcell), I(o_tcell), s));
    // 2. matchGrid with the stereo window (:141-143, :340-342: matching_s_ws cells to the left, same row)
    GridParams prm{rows, cols, CAP, mc->best_lr_matches ? 1 : 0, PlGridWindow{mc->matching_s_ws, 0, 0, 0}, mc->min_ratio_12_p,
                   mc->line_sim_th};
    CK(ctx, launch_match_grid(reinterpret_cast<GridProblem*>(base + o_prob), B, prm, lines, s));
    // 3. lifting, reading the match list where matchGrid left it
    if (lines)
        CK(ctx, launch_lift_lines(*cam, *sc, B, I(o_loff), F(o_xyl), F(o_ang), I(o_oct), base + o_d1, I(o_roff), F(o_xyr), I(o_m12),
                                  D(o_pl), D(o_epl), D(o_disp), D(o_edisp), D(o_P), D(o_eP), D(o_le), D(o_angd), D(o_s2), I(o_lvl),
                                  base + o_dout, I(o_src), I(o_cnt), s));
    else
        CK(ctx, launch_lift_points(*cam, *sc, B, I(o_loff), F(o_xyl), I(o_oct), base + o_d1, I(o_roff), F(o_xyr), I(o_m12), D(o_pl),
                                   D(o_disp), D(o_P), D(o_s2), I(o_lvl), base + o_dout, I(o_src), I(o_cnt), s));
    ctx->launches += 3;
    std::vector<int32_t> gcnt((size_t)B), cnt((size_t)B);
    CK(ctx, down(out.m12, o_m12, N1 * 4));
    CK(ctx, down(out.a_pl, o_pl, N1 * 16));
    CK(ctx, down(out.a_disp, o_disp, N1 * 8));
    CK(ctx, down(out.a_P, o_P, N1 * 24));
    CK(ctx, down(out.a_s2, o_s2, N1 * 8));
    CK(ctx, down(out.level, o_lvl, N1 * 4));
    CK(ctx, down(out.desc, o_dout, N1 * 32));
    CK(ctx, down(out.src, o_src, N1 * 4));
    if (lines) {
        CK(ctx, down(out.epl, o_epl, N1 * 16));
        CK(ctx, down(out.edisp, o_edisp, N1 * 8));
        CK(ctx, down(out.eP, o_eP, N1 * 24));
        CK(ctx, down(out.le, o_le, N1 * 24));
        CK(ctx, down(out.angle, o_angd, N1 * 8));
    }
    CK(ctx, down(gcnt.data(), o_gcnt, (size_t)B * 4));
    CK(ctx, down(cnt.data(), o_cnt, (size_t)B * 4));
    CK(ctx, cudaStreamSynchronize(s));
    long total = 0;
    for (int p = 0; p < B; ++p) {
        if (gcnt[p] < 0) return fail(ctx, gcnt[p], "matchGrid: more than 128 candidates in one query window");
        if (out.counts) out.counts[p] = cnt[p];
        total += cnt[p];
    }
    return (int)total;
}
}  // namespace

int plstvo_match_stereo_points(PlContext* ctx, const PlCamera* cam, const PlStereoMatchConfig* mcfg, const PlStereoConfig* scfg,
                               int B, const int32_t* l_off, const float* kp_l, const int32_t* octave_l, const uint8_t* desc_l,
                               const int32_t* r_off, const float* kp_r, const uint8_t* desc_r, int32_t* m12, double* pt_pl,
                               double* pt_disp, double* pt_P, double* pt_sigma2, int32_t* pt_level, uint8_t* pdesc_out,
                               int32_t* src_idx, int32_t* counts) {
    const StereoOut out{m12, pt_pl, pt_disp, pt_P, pt_sigma2, pt_level, pdesc_out, src_idx, counts,
                        nullptr, nullptr, nullptr, nullptr, nullptr};
    return match_stereo_common(ctx, false, cam, mcfg, scfg, B, l_off, kp_l, nullptr, octave_l, desc_l, r_off, kp_r, desc_r, out);
}

int plstvo_match_stereo_lines(PlContext* ctx, const PlCamera* cam, const PlStereoMatchConfig* mcfg, const PlStereoConfig* scfg,
                              int B, const int32_t* l_off, const float* seg_l, const float* angle_l, const int32_t* octave_l,
                              const uint8_t* desc_l, const int32_t* r_off, const float* seg_r, const uint8_t* desc_r,
                              int32_t* m12, double* ls_spl, double* ls_epl, double* ls_sdisp, double* ls_edisp, double* ls_sP,
                              double* ls_eP, double* ls_le, double* ls_angle, double* ls_sigma2, int32_t* ls_level,
                              uint8_t* ldesc_out, int32_t* src_idx, int32_t* counts) {
    const StereoOut out{m12, ls_spl, ls_sdisp, ls_sP, ls_sigma2, ls_level, ldesc_out, src_idx, counts,
                        ls_epl, ls_edisp, ls_eP, ls_le, ls_angle};
    return match_stereo_common(ctx, true, cam, mcfg, scfg, B, l_off, seg_l, angle_l, octave_l, desc_l, r_off, seg_r, desc_r, out);
}

// ---- raw stereo features -> pose, records resident in HBM ---------------------------------------------------------
// sequence == false: B independent (prev, curr) pairs, four feature sets of B frames.
// sequence == true : prev holds NF = B + 1 consecutive frames, pair p = (frame p, frame p + 1); two feature sets of NF frames,
//                    every frame goes through the stereo step once and is lifted twice (as a previous and as a current frame).
static int track_stereo_common(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg, const PlStereoMatchConfig* mc,
                               const PlStereoConfig* sc, const PlStereoFeatures* prev, const PlStereoFeatures* curr,
                               const PlPrior* priors, PlPoseResult* results, int32_t* n_stereo, bool sequence, int slot) {
    // slot < 0: blocking (returns with the results in host memory); slot 0 / 1: enqueue only, results valid after plstvo_wait
    if (!ctx) return PLSTVO_E_INVALID;
    LOCK(ctx);
    if (!cam || !cfg || !mc || !sc || !prev || (!sequence && !curr) || !results) return fail(ctx, PLSTVO_E_INVALID, "null argument");
    const int NF = prev->B;                         // frames per feature set
    const int B = sequence ? NF - 1 : NF;           // pairs
    if (NF < 0 || (!sequence && curr->B != NF)) return fail(ctx, PLSTVO_E_SIZE, "prev and curr hold different numbers of frames");
    if (sequence && NF == 1) return 0;              // one frame: nothing to track
    const int rows = mc->grid_rows, cols = mc->grid_cols;
    if (rows <= 0 || cols <= 0 || rows * cols > 8192 || cam->width <= 0 || cam->height <= 0)
        return fail(ctx, PLSTVO_E_INVALID, "bad grid or image size");
    if (NF == 0) return 0;
    CK(ctx, cudaSetDevice(ctx->device));
    constexpr int CAP = 128;
    const int NSETS = sequence ? 2 : 4;
    if (sequence) curr = prev;                      // sets 2, 3 below are unused
    // the four feature sets: {prev, curr} x {points, lines}
    struct Set {
        bool lines; const int32_t *l_off, *r_off; const float *xy_l, *xy_r, *ang; const int32_t* oct; const uint8_t *d1, *d2;
        size_t N1, N2, o_loff, o_roff, o_xyl, o_xyr, o_ang, o_oct, o_d1, o_d2, o_m12, o_cnt, o_gcnt, o_ooff, o_ooff2, o_prob;
    };
    Set sets[4] = {
        {false, prev->pl_off, prev->pr_off, prev->kp_l, prev->kp_r, nullptr, prev->poct_l, prev->pdesc_l, prev->pdesc_r},
        {true, prev->ll_off, prev->lr_off, prev->seg_l, prev->seg_r, prev->angle_l, prev->loct_l, prev->ldesc_l, prev->ldesc_r},
        {false, curr->pl_off, curr->pr_off, curr->kp_l, curr->kp_r, nullptr, curr->poct_l, curr->pdesc_l, curr->pdesc_r},
        {true, curr->ll_off, curr->lr_off, curr->seg_l, curr->seg_r, curr->angle_l, curr->loct_l, curr->ldesc_l, curr->ldesc_r}};
    LiftArena a;
    size_t maxN1 = 0, maxN2 = 0, max_items = 0;
    for (int k = 0; k < NSETS; ++k) {
        Set& st = sets[k];
        int rc = lift_check_offsets(ctx, NF, st.l_off, st.r_off);
        if (rc) return rc;
        st.N1 = st.l_off[NF];
        st.N2 = st.r_off[NF];
        if (st.N1 && (!st.xy_l || !st.oct || !st.d1 || (st.lines && !st.ang))) return fail(ctx, PLSTVO_E_INVALID, "null input array");
        if (st.N2 && (!st.xy_r || !st.d2)) return fail(ctx, PLSTVO_E_INVALID, "null input array");
        const int cw = st.lines ? 4 : 2;
        st.o_loff = a.take((size_t)(NF + 1) * 4); st.o_roff = a.take((size_t)(NF + 1) * 4);
        st.o_xyl = a.take(st.N1 * cw * 4); st.o_xyr = a.take(st.N2 * cw * 4); st.o_ang = a.take(st.lines ? st.N1 * 4 : 0);
        st.o_oct = a.take(st.N1 * 4); st.o_d1 = a.take(st.N1 * 32); st.o_d2 = a.take(st.N2 * 32); st.o_m12 = a.take(st.N1 * 4);
        st.o_cnt = a.take((size_t)NF * 4); st.o_gcnt = a.take((size_t)NF * 4); st.o_ooff = a.take((size_t)(NF + 1) * 4);
        st.o_ooff2 = a.take((size_t)(NF + 1) * 4);
        st.o_prob = a.take((size_t)NF * sizeof(GridProblem));
        maxN1 = std::max(maxN1, st.N1);
        maxN2 = std::max(maxN2, st.N2);
        max_items = std::max(max_items, st.N2 * (st.lines ? (size_t)std::max(rows, cols) + 2 : 1));
    }
    // matchGrid scratch, shared by the four sets (they run one after the other on one stream)
    const size_t o_qcell = a.take(maxN1 * 16), o_tcell = a.take(maxN2 * 8), o_tline = a.take(maxN2 * 32), o_tdir = a.take(maxN2 * 16);
    const size_t o_items = a.take(max_items * 4), o_qpairs = a.take(maxN1 * CAP * 8), o_qcount = a.take(maxN1 * 4);
    const size_t o_tcount = a.take(maxN2 * 4), o_tstart = a.take((maxN2 + NF) * 4), o_tslots = a.take(maxN1 * CAP * 4);
    const size_t o_seen = a.take(maxN1 * CAP), o_m21 = a.take(maxN2 * 4);
    DevBuf& arena = ctx->arena_track_stereo[slot + 1];
    CK(ctx, arena.ensure(a.off));
    uint8_t* base = arena.as<uint8_t>();
    auto I = [&](size_t o) { return reinterpret_cast<int32_t*>(base + o); };
    auto D = [&](size_t o) { return reinterpret_cast<double*>(base + o); };
    auto F = [&](size_t o) { return reinterpret_cast<float*>(base + o); };
    cudaStream_t s = ctx->s_main, sh = ctx->s_h2d;   // uploads of set k + 1 run under the kernels of set k
    auto up = [&](size_t o, const void* src, size_t bytes) -> cudaError_t {
        return (src && bytes) ? cudaMemcpyAsync(base + o, src, bytes, cudaMemcpyHostToDevice, sh) : cudaSuccess;
    };
    // (this slot's arena is free: a blocking call ends synchronised, an async slot is reused only after its event completed)
    const double inv_w = cols / static_cast<double>(cam->width), inv_h = rows / static_cast<double>(cam->height);
    const GridParams gprm{rows, cols, CAP, mc->best_lr_matches ? 1 : 0, PlGridWindow{mc->matching_s_ws, 0, 0, 0}, mc->min_ratio_12_p,
                          mc->line_sim_th};
    // pinned staging: 4 problem tables + 2 x 4 x B counters (pageable copies would block this thread on the stream)
    const size_t prob_bytes = ((size_t)NF * sizeof(GridProblem) + 255) / 256 * 256;
    CK(ctx, ctx->staging(slot + 1, 4 * prob_bytes + (size_t)8 * NF * 4));
    uint8_t* hst = static_cast<uint8_t*>(ctx->h_staging[slot + 1]);
    int32_t* cnt = reinterpret_cast<int32_t*>(hst + 4 * prob_bytes);
    int32_t* gcnt = cnt + (size_t)4 * NF;
    // ---- pass 1: cells -> matchGrid -> lifting filters (count only) per set ----
    for (int k = 0; k < NSETS; ++k) {
        Set& st = sets[k];
        const int cw = st.lines ? 4 : 2;
        const size_t per_train_cells = st.lines ? (size_t)std::max(rows, cols) + 2 : 1;
        GridProblem* probs = reinterpret_cast<GridProblem*>(hst + (size_t)k * prob_bytes);
        for (int p = 0; p < NF; ++p) {
            GridProblem& g = probs[p];
            const size_t qa = st.l_off[p], tb = st.r_off[p];
            g.n1 = st.l_off[p + 1] - st.l_off[p];
            g.n2 = st.r_off[p + 1] - st.r_off[p];
            g.q_cell = I(o_qcell) + qa * cw;
            g.d1 = base + st.o_d1 + qa * 32;
            g.t_cell = st.lines ? nullptr : I(o_tcell) + tb * 2;
            g.t_line = st.lines ? D(o_tline) + tb * 4 : nullptr;
            g.t_dir = st.lines ? D(o_tdir) + tb * 2 : nullptr;
            g.d2 = base + st.o_d2 + tb * 32;
            g.m12 = I(st.o_m12) + qa;
            g.count = I(st.o_gcnt) + p;
            g.grid_items = I(o_items) + tb * per_train_cells;
            g.q_pairs = reinterpret_cast<int2*>(base + o_qpairs) + qa * CAP;
            g.q_count = I(o_qcount) + qa;
            g.t_count = I(o_tcount) + tb;
            g.t_start = I(o_tstart) + tb + p;
            g.t_slots = I(o_tslots) + qa * CAP;
            g.seen = base + o_seen + qa * CAP;
            g.m21 = I(o_m21) + tb;
        }
        CK(ctx, up(st.o_loff, st.l_off, (size_t)(NF + 1) * 4));
        CK(ctx, up(st.o_roff, st.r_off, (size_t)(NF + 1) * 4));
        CK(ctx, up(st.o_xyl, st.xy_l, st.N1 * cw * 4));
        CK(ctx, up(st.o_xyr, st.xy_r, st.N2 * cw * 4));
        if (st.lines) CK(ctx, up(st.o_ang, st.ang, st.N1 * 4));
        CK(ctx, up(st.o_oct, st.oct, st.N1 * 4));
        CK(ctx, up(st.o_d1, st.d1, st.N1 * 32));
        CK(ctx, up(st.o_d2, st.d2, st.N2 * 32));
        CK(ctx, up(st.o_prob, probs, (size_t)NF * sizeof(GridProblem)));
        cudaEvent_t uploaded = next_event(ctx);
        CK(ctx, cudaEventRecord(uploaded, sh));
        CK(ctx, cudaStreamWaitEvent(s, uploaded, 0));
        if (st.lines) {
            CK(ctx, launch_stereo_cells_lines((int)st.N1, (int)st.N2, inv_w, inv_h, F(st.o_xyl), F(st.o_xyr), I(o_qcell), D(o_tline),
                                              D(o_tdir), s));
            CK(ctx, launch_match_grid(reinterpret_cast<GridProblem*>(base + st.o_prob), NF, gprm, true, s));
            CK(ctx, launch_lift_lines(*cam, *sc, NF, I(st.o_loff), F(st.o_xyl), F(st.o_ang), I(st.o_oct), base + st.o_d1, I(st.o_roff),
                                      F(st.o_xyr), I(st.o_m12), nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                                      nullptr, nullptr, nullptr, nullptr, I(st.o_cnt), s));
        } else {
            CK(ctx, launch_stereo_cells_points((int)st.N1, (int)st.N2, inv_w, inv_h, F(st.o_xyl), F(st.o_xyr), I(o_qcell), I(o_tcell), s));
            CK(ctx, launch_match_grid(reinterpret_cast<GridProblem*>(base + st.o_prob), NF, gprm, false, s));
            CK(ctx, launch_lift_points(*cam, *sc, NF, I(st.o_loff), F(st.o_xyl), I(st.o_oct), base + st.o_d1, I(st.o_roff), F(st.o_xyr),
                                       I(st.o_m12), nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, I(st.o_cnt), s));
        }
        ctx->launches += 3;
        CK(ctx, cudaMemcpyAsync(cnt + (size_t)k * NF, base + st.o_cnt, (size_t)NF * 4, cudaMemcpyDeviceToHost, s));
        CK(ctx, cudaMemcpyAsync(gcnt + (size_t)k * NF, base + st.o_gcnt, (size_t)NF * 4, cudaMemcpyDeviceToHost, s));
    }
    CK(ctx, cudaStreamSynchronize(s));     // the one host hop: survivor counts -> compact offsets and the matcher's tile plan
    // compact offsets per set; in sequence mode the current-frame role of a set starts at its second frame
    std::vector<int32_t> ooff[4], ooff2[2];
    for (int k = 0; k < NSETS; ++k) {
        ooff[k].assign((size_t)NF + 1, 0);
        for (int p = 0; p < NF; ++p) {
            if (gcnt[(size_t)k * NF + p] < 0) return fail(ctx, gcnt[(size_t)k * NF + p], "matchGrid: more than 128 candidates in one query window");
            ooff[k][p + 1] = ooff[k][p] + cnt[(size_t)k * NF + p];
            if (n_stereo) {
                if (sequence) n_stereo[(size_t)p * 2 + k] = cnt[(size_t)k * NF + p];
                else n_stereo[(size_t)p * 4 + k] = cnt[(size_t)k * NF + p];
            }
        }
        CK(ctx, up(sets[k].o_ooff, ooff[k].data(), (size_t)(NF + 1) * 4));
        if (sequence) {
            ooff2[k].assign((size_t)NF, 0);          // frames 1 .. NF - 1 as current frames: offsets relative to frame 1
            for (int p = 0; p < NF; ++p) ooff2[k][p] = ooff[k][p + 1] - ooff[k][1];
            CK(ctx, up(sets[k].o_ooff2, ooff2[k].data(), (size_t)NF * 4));
        }
    }
    // ---- the tracker's plan on the compact lists; the records are written straight into its buffers ----
    PlFrameBatch fp{}, fc{};
    fp.B = fc.B = B;
    fp.pt_off = ooff[0].data(); fp.ls_off = ooff[1].data();
    fc.pt_off = sequence ? ooff2[0].data() : ooff[2].data();
    fc.ls_off = sequence ? ooff2[1].data() : ooff[3].data();
    Workspace& ws = slot < 0 ? ctx->ws : ctx->ws_async[slot];
    int rc = ws_prepare(ctx, ws, cam, cfg, &fp, &fc, true, priors != nullptr);
    if (rc) return rc;
    if (priors) CK(ctx, cudaMemcpyAsync(ws.d_priors.p, priors, (size_t)B * sizeof(PlPrior), cudaMemcpyHostToDevice, ctx->s_h2d));
    cudaEvent_t planned = next_event(ctx);
    CK(ctx, cudaEventRecord(planned, ctx->s_h2d));
    CK(ctx, cudaStreamWaitEvent(s, planned, 0));
    // pass 2: the same lifting kernels, now writing at the compact offsets (prev role: P, sigma2, segments, level; curr role: pl, le).
    // `first` = first frame of the role inside its set (sequence mode: the current-frame role starts at frame 1).
    auto lift_prev_points = [&](const Set& st) -> cudaError_t {
        return launch_lift_points(*cam, *sc, B, I(st.o_loff), F(st.o_xyl), I(st.o_oct), base + st.o_d1, I(st.o_roff), F(st.o_xyr),
                                  I(st.o_m12), nullptr, nullptr, ws.d_ptP.as<double>(), ws.d_pts2.as<double>(), nullptr,
                                  ws.d_pdesc1.as<uint8_t>(), nullptr, I(st.o_cnt), s, I(st.o_ooff));
    };
    auto lift_prev_lines = [&](const Set& st) -> cudaError_t {
        return launch_lift_lines(*cam, *sc, B, I(st.o_loff), F(st.o_xyl), F(st.o_ang), I(st.o_oct), base + st.o_d1, I(st.o_roff),
                                 F(st.o_xyr), I(st.o_m12), ws.d_lsspl.as<double>(), ws.d_lsepl.as<double>(), nullptr, nullptr,
                                 ws.d_lssP.as<double>(), ws.d_lseP.as<double>(), nullptr, nullptr, ws.d_lss2.as<double>(),
                                 ws.d_lslev.as<int32_t>(), ws.d_ldesc1.as<uint8_t>(), nullptr, I(st.o_cnt), s, I(st.o_ooff));
    };
    auto lift_curr_points = [&](const Set& st, int first, size_t o_out) -> cudaError_t {
        return launch_lift_points(*cam, *sc, B, I(st.o_loff) + first, F(st.o_xyl), I(st.o_oct), base + st.o_d1, I(st.o_roff) + first,
                                  F(st.o_xyr), I(st.o_m12), ws.d_ptpl.as<double>(), nullptr, nullptr, nullptr, nullptr,
                                  ws.d_pdesc2.as<uint8_t>(), nullptr, I(st.o_cnt) + first, s, I(o_out));
    };
    auto lift_curr_lines = [&](const Set& st, int first, size_t o_out) -> cudaError_t {
        return launch_lift_lines(*cam, *sc, B, I(st.o_loff) + first, F(st.o_xyl), F(st.o_ang), I(st.o_oct), base + st.o_d1,
                                 I(st.o_roff) + first, F(st.o_xyr), I(st.o_m12), nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                                 ws.d_lsle.as<double>(), nullptr, nullptr, nullptr, ws.d_ldesc2.as<uint8_t>(), nullptr,
                                 I(st.o_cnt) + first, s, I(o_out));
    };
    CK(ctx, lift_prev_points(sets[0]));
    CK(ctx, lift_prev_lines(sets[1]));
    if (sequence) {
        CK(ctx, lift_curr_points(sets[0], 1, sets[0].o_ooff2));
        CK(ctx, lift_curr_lines(sets[1], 1, sets[1].o_ooff2));
    } else {
        CK(ctx, lift_curr_points(sets[2], 0, sets[2].o_ooff));
        CK(ctx, lift_curr_lines(sets[3], 0, sets[3].o_ooff));
    }
    ctx->launches += 4;
    rc = ws_launch_match(ctx, ws, 0, B, s);
    if (rc) return rc;
    rc = ws_launch_solve(ctx, ws, 0, B, true, s);
    if (rc) return rc;
    CK(ctx, cudaMemcpyAsync(results, ws.d_results.p, (size_t)B * sizeof(PlPoseResult), cudaMemcpyDeviceToHost, s));
    if (slot < 0) CK(ctx, cudaStreamSynchronize(s));
    return 0;
}

// ticket bookkeeping shared with plstvo_track_batch_async: two slots, plstvo_wait(ticket) blocks until the slot's results are home
static int stereo_async(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg, const PlStereoMatchConfig* mc,
                        const PlStereoConfig* sc, const PlStereoFeatures* a, const PlStereoFeatures* b, const PlPrior* priors,
                        PlPoseResult* results, int32_t* n_stereo, bool sequence) {
    if (!ctx) return PLSTVO_E_INVALID;
    LOCK(ctx);
    CK(ctx, cudaSetDevice(ctx->device));
    const int slot = ctx->next_slot;
    ctx->next_slot ^= 1;
    if (ctx->slot_busy[slot]) {
        CK(ctx, cudaEventSynchronize(ctx->slot_done[slot]));
        ctx->slot_busy[slot] = false;
    }
    if (!ctx->slot_done[slot]) CK(ctx, cudaEventCreateWithFlags(&ctx->slot_done[slot], cudaEventDisableTiming));
    const int rc = track_stereo_common(ctx, cam, cfg, mc, sc, a, b, priors, results, n_stereo, sequence, slot);
    if (rc) return rc;
    CK(ctx, cudaEventRecord(ctx->slot_done[slot], ctx->s_main));
    ctx->slot_busy[slot] = true;
    return slot;
}

int plstvo_track_stereo_batch_async(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg, const PlStereoMatchConfig* mc,
                                    const PlStereoConfig* sc, const PlStereoFeatures* prev, const PlStereoFeatures* curr,
                                    const PlPrior* priors, PlPoseResult* results, int32_t* n_stereo) {
    return stereo_async(ctx, cam, cfg, mc, sc, prev, curr, priors, results, n_stereo, false);
}

int plstvo_track_stereo_sequence_async(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg, const PlStereoMatchConfig* mc,
                                       const PlStereoConfig* sc, const PlStereoFeatures* frames, const PlPrior* priors,
                                       PlPoseResult* results, int32_t* n_stereo) {
    return stereo_async(ctx, cam, cfg, mc, sc, frames, nullptr, priors, results, n_stereo, true);
}

int plstvo_track_stereo_batch(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg, const PlStereoMatchConfig* mc,
                              const PlStereoConfig* sc, const PlStereoFeatures* prev, const PlStereoFeatures* curr,
                              const PlPrior* priors, PlPoseResult* results, int32_t* n_stereo) {
    return track_stereo_common(ctx, cam, cfg, mc, sc, prev, curr, priors, results, n_stereo, false, -1);
}

int plstvo_track_stereo_sequence(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg, const PlStereoMatchConfig* mc,
                                 const PlStereoConfig* sc, const PlStereoFeatures* frames, const PlPrior* priors,
                                 PlPoseResult* results, int32_t* n_stereo) {
    return track_stereo_common(ctx, cam, cfg, mc, sc, frames, nullptr, priors, results, n_stereo, true, -1);
}

// ---- stereoFrameHandler.h surface ------------------------------------------------------------------------
int plstvo_f2f_tracking(PlContext* ctx, const PlConfig* cfg, const PlFrameBatch* prev, const PlFrameBatch* curr,
                        int32_t* m12_pt, int32_t* m12_ls, int32_t* n_matched) {
    if (!ctx || !cfg) return PLSTVO_E_INVALID;
    LOCK(ctx);
    CK(ctx, cudaSetDevice(ctx->device));
    int rc = validate_frames(ctx, prev, curr, false);
    if (rc) return rc;
    const int B = prev->B;
    if (B == 0) return 0;
    Workspace& ws = ctx->ws;
    rc = ws_prepare(ctx, ws, nullptr, cfg, prev, curr, false, false);
    if (rc) return rc;
    rc = ws_upload_range(ctx, ws, prev, curr, nullptr, 0, B, false, ctx->s_h2d);
    if (rc) return rc;
    cudaEvent_t up = next_event(ctx);
    CK(ctx, cudaEventRecord(up, ctx->s_h2d));
    CK(ctx, cudaStreamWaitEvent(ctx->s_main, up, 0));
    rc = ws_launch_match(ctx, ws, 0, B, ctx->s_main);
    if (rc) return rc;
    CK(ctx, ctx->scratch.ensure((size_t)2 * B * 4));
    CK(ctx, launch_match_finalize(ws.d_problems.as<MatchProblem>(), 2 * B, ws.max_n2, ctx->scratch.as<int32_t>(),
                                  ctx->s_main));
    ctx->launches++;
    if (m12_pt && prev->pt_off[B])
        CK(ctx, cudaMemcpyAsync(m12_pt, ws.d_m12p.p, (size_t)prev->pt_off[B] * 4, cudaMemcpyDeviceToHost, ctx->s_main));
    if (m12_ls && prev->ls_off[B])
        CK(ctx, cudaMemcpyAsync(m12_ls, ws.d_m12l.p, (size_t)prev->ls_off[B] * 4, cudaMemcpyDeviceToHost, ctx->s_main));
    if (n_matched)
        CK(ctx, cudaMemcpyAsync(n_matched, ctx->scratch.p, (size_t)2 * B * 4, cudaMemcpyDeviceToHost, ctx->s_main));
    CK(ctx, cudaStreamSynchronize(ctx->s_main));
    return 0;
}

int plstvo_optimize_pose(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg, const PlMatchedBatch* m,
                         const PlPrior* priors, PlPoseResult* results, uint8_t* inlier_pt, uint8_t* inlier_ls) {
    if (!ctx || !cam || !cfg || !m || !results) return PLSTVO_E_INVALID;
    LOCK(ctx);
    const int B = m->B;
    if (B < 0) return fail(ctx, PLSTVO_E_INVALID, "negative batch size");
    if (B == 0) return 0;
    if (!m->pt_off || !m->ls_off) return fail(ctx, PLSTVO_E_INVALID, "null offsets");
    CK(ctx, cudaSetDevice(ctx->device));
    int cap_pt = 1, cap_ls = 1;
    for (int p = 0; p < B; ++p) {
        const int n = m->pt_off[p + 1] - m->pt_off[p], l = m->ls_off[p + 1] - m->ls_off[p];
        if (n < 0 || l < 0) return fail(ctx, PLSTVO_E_INVALID, "offsets are not non-decreasing");
        if (n > PLSTVO_MAX_FEATURES || l > PLSTVO_MAX_FEATURES) return fail(ctx, PLSTVO_E_TOO_LARGE, "list too long");
        cap_pt = std::max(cap_pt, n);
        cap_ls = std::max(cap_ls, l);
    }
    const size_t n = m->pt_off[B], l = m->ls_off[B];
    if (n && (!m->pt_P || !m->pt_pl_obs || !m->pt_sigma2)) return fail(ctx, PLSTVO_E_INVALID, "point arrays missing");
    if (l && (!m->ls_sP || !m->ls_eP || !m->ls_le_obs || !m->ls_spl || !m->ls_epl || !m->ls_sigma2))
        return fail(ctx, PLSTVO_E_INVALID, "line arrays missing");
    const int sort_cap = pow2_ceil_host(std::max(32, std::max(cap_pt, cap_ls)));
    bool in_smem = getenv("PLSTVO_K2_FEAT_GLOBAL") == nullptr && k2_smem_bytes(cap_pt, cap_ls, sort_cap, true) <= ctx->smem_optin;
    if (!in_smem && k2_smem_bytes(cap_pt, cap_ls, sort_cap, false) > ctx->smem_optin)
        return fail(ctx, PLSTVO_E_TOO_LARGE, "lists too long for the per-pair solver's shared memory");

    Workspace& ws = ctx->ws;
    ws.planned = false;   // the explicit-list path reuses the workspace's buffers with its own layout
    cudaStream_t s = ctx->s_main;
    struct Up { DevBuf* buf; const void* src; size_t bytes; };
    Up ups[] = {{&ws.d_poff1, m->pt_off, (size_t)(B + 1) * 4}, {&ws.d_loff1, m->ls_off, (size_t)(B + 1) * 4},
                {&ws.d_ptP, m->pt_P, n * 24}, {&ws.d_ptpl, m->pt_pl_obs, n * 16}, {&ws.d_pts2, m->pt_sigma2, n * 8},
                {&ws.d_inlp, m->pt_inlier, n}, {&ws.d_lssP, m->ls_sP, l * 24}, {&ws.d_lseP, m->ls_eP, l * 24},
                {&ws.d_lsle, m->ls_le_obs, l * 24}, {&ws.d_lsspl, m->ls_spl, l * 16}, {&ws.d_lsepl, m->ls_epl, l * 16},
                {&ws.d_lss2, m->ls_sigma2, l * 8}, {&ws.d_inll, m->ls_inlier, l}};
    for (auto& u : ups) {
        CK(ctx, u.buf->ensure(std::max<size_t>(u.bytes, 16)));
        if (u.src && u.bytes) CK(ctx, cudaMemcpyAsync(u.buf->p, u.src, u.bytes, cudaMemcpyHostToDevice, s));
    }
    CK(ctx, ws.d_results.ensure((size_t)B * sizeof(PlPoseResult)));
    CK(ctx, ws.d_priors.ensure((size_t)B * sizeof(PlPrior)));
    if (priors) CK(ctx, cudaMemcpyAsync(ws.d_priors.p, priors, (size_t)B * sizeof(PlPrior), cudaMemcpyHostToDevice, s));
    // output flags live in separate buffers (the input flags are read while the outputs are written)
    CK(ctx, ctx->gn_out[0].ensure(std::max<size_t>(n, 16)));
    CK(ctx, ctx->gn_out[1].ensure(std::max<size_t>(l, 16)));
    size_t stride = 0;
    const bool streamed = stream_mode() == 1 || (stream_mode() != 0 && (!in_smem || (B > ctx->sm_count && cfg->solver_mode == 0)));
    if (!in_smem || streamed) {
        stride = k2_feat_stride(cap_pt, cap_ls);
        CK(ctx, ws.d_feat.ensure((size_t)B * stride * sizeof(double)));
    }
    SolveParams prm{};
    prm.cam = *cam;
    prm.cfg = *cfg;
    prm.mode = 1;
    prm.first_pair = 0;
    prm.matched = MatchedDev{ws.d_poff1.as<int32_t>(), ws.d_loff1.as<int32_t>(), ws.d_ptP.as<double>(),
                             ws.d_ptpl.as<double>(), ws.d_pts2.as<double>(),
                             m->pt_inlier ? ws.d_inlp.as<uint8_t>() : nullptr, ws.d_lssP.as<double>(),
                             ws.d_lseP.as<double>(), ws.d_lsle.as<double>(), ws.d_lsspl.as<double>(),
                             ws.d_lsepl.as<double>(), ws.d_lss2.as<double>(),
                             m->ls_inlier ? ws.d_inll.as<uint8_t>() : nullptr};
    prm.priors = priors ? ws.d_priors.as<PlPrior>() : nullptr;
    prm.results = ws.d_results.as<PlPoseResult>();
    prm.inlier_pt = ctx->gn_out[0].as<uint8_t>();
    prm.inlier_ls = ctx->gn_out[1].as<uint8_t>();
    prm.feat_scratch = in_smem ? nullptr : ws.d_feat.as<double>();
    prm.feat_scratch_stride = stride;
    prm.cap_pt = cap_pt;
    prm.cap_ls = cap_ls;
    prm.sort_cap = sort_cap;
    prm.feat_in_smem = in_smem ? 1 : 0;
    if (streamed) {
        StreamBufs sb;
        const int rc = stream_bufs_prepare(ctx, ws.d_stream, B, n, l, &sb);
        if (rc) return rc;
        prm.feat_scratch = ws.d_feat.as<double>();
        prm.feat_in_smem = 0;
        int nl = 0;
        CK(ctx, launch_stream_solve(prm, B, sb, s, &nl));
        ctx->launches += nl;
    } else {
        CK(ctx, launch_track_solve(prm, B, s));
        ctx->launches++;
    }
    CK(ctx, cudaMemcpyAsync(results, ws.d_results.p, (size_t)B * sizeof(PlPoseResult), cudaMemcpyDeviceToHost, s));
    if (inlier_pt && n) CK(ctx, cudaMemcpyAsync(inlier_pt, ctx->gn_out[0].p, n, cudaMemcpyDeviceToHost, s));
    if (inlier_ls && l) CK(ctx, cudaMemcpyAsync(inlier_ls, ctx->gn_out[1].p, l, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    return 0;
}

// enqueue one batch on the context's streams: chunked H2D -> K1 -> K2 -> D2H, nothing is waited for
static int track_enqueue(PlContext* ctx, Workspace& ws, const PlCamera* cam, const PlConfig* cfg,
                         const PlFrameBatch* prev, const PlFrameBatch* curr, const PlPrior* priors,
                         PlPoseResult* results, int32_t* m12_pt, int32_t* m12_ls, uint8_t* inlier_pt,
                         uint8_t* inlier_ls, bool pipelined) {
    const int B = prev->B;
    int rc = ws_prepare(ctx, ws, cam, cfg, prev, curr, true, priors != nullptr);
    if (rc) return rc;
    const bool have_level = prev->ls_level != nullptr;
    const std::vector<int> bounds = chunk_schedule(B, ctx->sm_count, pipelined);
    for (int k = 0; k + 1 < (int)bounds.size(); ++k) {
        const int p0 = bounds[k], p1 = bounds[k + 1];
        rc = ws_upload_range(ctx, ws, prev, curr, priors, p0, p1, true, ctx->s_h2d);
        if (rc) return rc;
        cudaEvent_t up = next_event(ctx);
        CK(ctx, cudaEventRecord(up, ctx->s_h2d));
        cudaStream_t s = (k & 1) ? ctx->s_alt : ctx->s_main;
        CK(ctx, cudaStreamWaitEvent(s, up, 0));
        rc = ws_launch_match(ctx, ws, p0, p1, s);
        if (rc) return rc;
        rc = ws_launch_solve(ctx, ws, p0, p1, have_level, s);
        if (rc) return rc;
        cudaEvent_t done = next_event(ctx);
        CK(ctx, cudaEventRecord(done, s));
        CK(ctx, cudaStreamWaitEvent(ctx->s_d2h, done, 0));
        rc = ws_download_range(ctx, ws, p0, p1, results, m12_pt, m12_ls, inlier_pt, inlier_ls, ctx->s_d2h);
        if (rc) return rc;
    }
    return 0;
}

int plstvo_track_batch(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg, const PlFrameBatch* prev,
                       const PlFrameBatch* curr, const PlPrior* priors, PlPoseResult* results, int32_t* m12_pt,
                       int32_t* m12_ls, uint8_t* inlier_pt, uint8_t* inlier_ls) {
    if (!ctx || !cam || !cfg) return PLSTVO_E_INVALID;
    LOCK(ctx);
    CK(ctx, cudaSetDevice(ctx->device));
    int rc = validate_frames(ctx, prev, curr, true);
    if (rc) return rc;
    if (prev->B == 0) return 0;
    rc = track_enqueue(ctx, ctx->ws, cam, cfg, prev, curr, priors, results, m12_pt, m12_ls, inlier_pt, inlier_ls, false);
    if (rc) return rc;
    CK(ctx, cudaStreamSynchronize(ctx->s_d2h));   // every chunk's D2H waited for its compute, which waited for its H2D
    return 0;
}

int plstvo_track_batch_async(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg, const PlFrameBatch* prev,
                             const PlFrameBatch* curr, const PlPrior* priors, PlPoseResult* results, int32_t* m12_pt,
                             int32_t* m12_ls, uint8_t* inlier_pt, uint8_t* inlier_ls) {
    if (!ctx || !cam || !cfg) return PLSTVO_E_INVALID;
    LOCK(ctx);
    CK(ctx, cudaSetDevice(ctx->device));
    int rc = validate_frames(ctx, prev, curr, true);
    if (rc) return rc;
    const int slot = ctx->next_slot;
    ctx->next_slot ^= 1;
    if (ctx->slot_busy[slot]) {   // the caller skipped plstvo_wait on the batch that used this slot: finish it first
        CK(ctx, cudaEventSynchronize(ctx->slot_done[slot]));
        ctx->slot_busy[slot] = false;
    }
    if (!ctx->slot_done[slot]) CK(ctx, cudaEventCreateWithFlags(&ctx->slot_done[slot], cudaEventDisableTiming));
    if (prev->B > 0) {
        rc = track_enqueue(ctx, ctx->ws_async[slot], cam, cfg, prev, curr, priors, results, m12_pt, m12_ls, inlier_pt,
                           inlier_ls, getenv("PLSTVO_ASYNC_RAMP") == nullptr);
        if (rc) return rc;
    }
    CK(ctx, cudaEventRecord(ctx->slot_done[slot], ctx->s_d2h));
    ctx->slot_busy[slot] = true;
    return slot;
}

int plstvo_wait(PlContext* ctx, int ticket) {
    if (!ctx || ticket < 0 || ticket > 1) return PLSTVO_E_INVALID;
    cudaEvent_t ev = nullptr;
    {
        LOCK(ctx);
        CK(ctx, cudaSetDevice(ctx->device));
        if (ctx->slot_busy[ticket]) ev = ctx->slot_done[ticket];
    }
    if (ev) {   // wait outside the lock: other threads may keep enqueueing on this context
        const cudaError_t e = cudaEventSynchronize(ev);
        LOCK(ctx);   // ctx->err is only ever written under the lock
        CK(ctx, e);
        ctx->slot_busy[ticket] = false;
    }
    return 0;
}

// ---- throughput mode ----------------------------------------------------------------------------------
int plstvo_batch_upload(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg, const PlFrameBatch* prev,
                        const PlFrameBatch* curr, const PlPrior* priors, PlDeviceBatch** out) {
    if (!ctx || !cam || !cfg || !out) return PLSTVO_E_INVALID;
    LOCK(ctx);
    *out = nullptr;
    CK(ctx, cudaSetDevice(ctx->device));
    int rc = validate_frames(ctx, prev, curr, true);
    if (rc) return rc;
    PlDeviceBatch* db = new PlDeviceBatch();
    rc = ws_prepare(ctx, db->ws, cam, cfg, prev, curr, true, priors != nullptr);
    if (rc == 0 && prev->B > 0) rc = ws_upload_range(ctx, db->ws, prev, curr, priors, 0, prev->B, true, ctx->s_h2d);
    if (rc == 0) {
        cudaError_t e = cudaStreamSynchronize(ctx->s_h2d);
        if (e != cudaSuccess) {
            ctx->err = cudaGetErrorString(e);
            rc = PLSTVO_E_CUDA;
        }
    }
    if (rc) {
        db->ws.release();
        delete db;
        return rc;
    }
    db->ws.have_level = prev->ls_level != nullptr;
    *out = db;
    return 0;
}

int plstvo_batch_run(PlContext* ctx, PlDeviceBatch* db) {
    if (!ctx || !db) return PLSTVO_E_INVALID;
    LOCK(ctx);
    CK(ctx, cudaSetDevice(ctx->device));
    return ws_run(ctx, db->ws, db->ws.have_level);
}

int plstvo_batch_run_timed(PlContext* ctx, PlDeviceBatch* db, int iters, int flush_l2, float* ms_total) {
    if (!ctx || !db || iters <= 0 || !ms_total) return PLSTVO_E_INVALID;
    LOCK(ctx);
    CK(ctx, cudaSetDevice(ctx->device));
    const size_t flush_bytes = 256u << 20;
    if (flush_l2) CK(ctx, ctx->scratch.ensure(flush_bytes));
    cudaEvent_t e0, e1;
    CK(ctx, cudaEventCreate(&e0));
    CK(ctx, cudaEventCreate(&e1));
    double total = 0.0;
    CK(ctx, cudaStreamSynchronize(ctx->s_main));
    if (!flush_l2) {
        CK(ctx, cudaEventRecord(e0, ctx->s_main));
        for (int i = 0; i < iters; ++i) {
                    int rc = ws_run(ctx, db->ws, db->ws.have_level);
            if (rc) return rc;
        }
        CK(ctx, cudaEventRecord(e1, ctx->s_main));
        CK(ctx, cudaEventSynchronize(e1));
        float ms = 0.f;
        CK(ctx, cudaEventElapsedTime(&ms, e0, e1));
        total = ms;
    } else {
        for (int i = 0; i < iters; ++i) {
            CK(ctx, cudaMemsetAsync(ctx->scratch.p, i & 0xFF, flush_bytes, ctx->s_main));
            CK(ctx, cudaEventRecord(e0, ctx->s_main));
                    int rc = ws_run(ctx, db->ws, db->ws.have_level);
            if (rc) return rc;
            CK(ctx, cudaEventRecord(e1, ctx->s_main));
            CK(ctx, cudaEventSynchronize(e1));
            float ms = 0.f;
            CK(ctx, cudaEventElapsedTime(&ms, e0, e1));
            total += ms;
        }
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *ms_total = (float)total;
    return 0;
}

int plstvo_batch_kernel_times(PlContext* ctx, PlDeviceBatch* db, int iters, double* ms_match, double* ms_solve,
                              int32_t* n_tiles, int32_t* n_pairs) {
    if (!ctx || !db || iters <= 0) return PLSTVO_E_INVALID;
    LOCK(ctx);
    CK(ctx, cudaSetDevice(ctx->device));
    Workspace& ws = db->ws;
    cudaEvent_t e0, e1, e2;
    CK(ctx, cudaEventCreate(&e0));
    CK(ctx, cudaEventCreate(&e1));
    CK(ctx, cudaEventCreate(&e2));
    double tm = 0.0, tsv = 0.0;
    const bool lev = ws.have_level;
    for (int i = 0; i < iters; ++i) {
        CK(ctx, cudaEventRecord(e0, ctx->s_main));
        int rc = ws_launch_match(ctx, ws, 0, ws.B, ctx->s_main);
        if (rc) return rc;
        CK(ctx, cudaEventRecord(e1, ctx->s_main));
        rc = ws_launch_solve(ctx, ws, 0, ws.B, lev, ctx->s_main);
        if (rc) return rc;
        CK(ctx, cudaEventRecord(e2, ctx->s_main));
        CK(ctx, cudaEventSynchronize(e2));
        float a = 0.f, b = 0.f;
        CK(ctx, cudaEventElapsedTime(&a, e0, e1));
        CK(ctx, cudaEventElapsedTime(&b, e1, e2));
        tm += a;
        tsv += b;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaEventDestroy(e2);
    if (getenv("PLSTVO_PHASE_DEBUG") && ws.B > 0) {   // per-phase device cycles of K2, averaged over the pairs
        CK(ctx, ws.d_phase.ensure((size_t)ws.B * 8 * sizeof(long long)));
        int rc2 = ws_launch_solve(ctx, ws, 0, ws.B, lev, ctx->s_main);
        if (rc2) return rc2;
        std::vector<long long> h((size_t)ws.B * 8);
        CK(ctx, cudaMemcpyAsync(h.data(), ws.d_phase.p, h.size() * sizeof(long long), cudaMemcpyDeviceToHost, ctx->s_main));
        CK(ctx, cudaStreamSynchronize(ctx->s_main));
        static const char* names[8] = {"match_finalize", "gather", "gn_eval", "gn_serial", "gates_eig", "outliers", "final", "sort_mad"};
        for (int k = 0; k < 8; ++k) {
            double sum = 0;
            for (int p = 0; p < ws.B; ++p) sum += (double)h[(size_t)p * 8 + k];
            fprintf(stderr, "[plstvo phase] %-15s %10.0f cycles/pair\n", names[k], sum / ws.B);
        }
        ws.d_phase.release();
    }
    if (ms_match) *ms_match = tm / iters;
    if (ms_solve) *ms_solve = tsv / iters;
    if (n_tiles)   // one tile per enabled matching problem
        *n_tiles = (int32_t)std::count_if(ws.problems.begin(), ws.problems.end(),
                                          [](const MatchProblem& pr) { return pr.enabled != 0; });
    if (n_pairs) *n_pairs = ws.B;
    return 0;
}

int plstvo_batch_stage_times(PlContext* ctx, PlDeviceBatch* db, int iters, double ms[8], int32_t counts[4]) {
    if (!ctx || !db || iters <= 0 || !ms) return PLSTVO_E_INVALID;
    LOCK(ctx);
    CK(ctx, cudaSetDevice(ctx->device));
    Workspace& ws = db->ws;
    // events: 0 start, 1 expand done, 2 distance done, 3 match done, 4 lists done, 5 GN stage 1 done, 6 outlier pass done,
    // 7 GN stage 2 done, 8 end
    cudaEvent_t ev[9];
    for (auto& e : ev) CK(ctx, cudaEventCreate(&e));
    double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = 0; i < iters; ++i) {
        CK(ctx, cudaEventRecord(ev[0], ctx->s_main));
        int rc = ws_launch_match(ctx, ws, 0, ws.B, ctx->s_main, &ev[1]);
        if (rc) return rc;
        CK(ctx, cudaEventRecord(ev[3], ctx->s_main));
        rc = ws_launch_solve(ctx, ws, 0, ws.B, ws.have_level, ctx->s_main, &ev[4]);
        if (rc) return rc;
        CK(ctx, cudaEventRecord(ev[8], ctx->s_main));
        CK(ctx, cudaEventSynchronize(ev[8]));
        auto span = [&](int a, int b, double& out) -> int {
            float t = 0.f;
            CK(ctx, cudaEventElapsedTime(&t, ev[a], ev[b]));
            out += t;
            return 0;
        };
        for (int k = 0; k < 4; ++k)
            if ((rc = span(k, k + 1, acc[k]))) return rc;
        if ((rc = span(4, 8, acc[4])) || (rc = span(4, 5, acc[5])) || (rc = span(5, 6, acc[6])) || (rc = span(6, 7, acc[7]))) return rc;
    }
    for (auto& e : ev) cudaEventDestroy(e);
    for (int k = 0; k < 8; ++k) ms[k] = acc[k] / iters;
    if (counts) {
        int delegated = 0;   // streamed solver: problems it handed to the fp64 kernel in the last pass (its only_if list)
        if (ws.use_stream && ws.B > 0) {
            StreamBufs sb;
            int rc = stream_bufs_prepare(ctx, ws.d_stream, ws.B, (size_t)ws.p_off1[ws.B], (size_t)ws.l_off1[ws.B], &sb);
            if (rc) return rc;
            std::vector<int32_t> act((size_t)ws.B);
            CK(ctx, cudaMemcpy(act.data(), sb.active, (size_t)ws.B * sizeof(int32_t), cudaMemcpyDeviceToHost));
            for (int32_t a : act) delegated += a != 0;
        }
        counts[0] = 1 | (ws.use_stream ? 2 : 0) | (delegated << 8);   // bit 0: tensor-core matcher (always)
        counts[1] = (int32_t)(ws.tc_items[0].size() + ws.tc_items[1].size());
        counts[2] = (int32_t)ws.problems.size();
        counts[3] = ws.B;
    }
    return 0;
}

int plstvo_batch_download(PlContext* ctx, PlDeviceBatch* db, PlPoseResult* results, int32_t* m12_pt,
                          int32_t* m12_ls, uint8_t* inlier_pt, uint8_t* inlier_ls) {
    if (!ctx || !db) return PLSTVO_E_INVALID;
    LOCK(ctx);
    CK(ctx, cudaSetDevice(ctx->device));
    if (db->ws.B == 0) return 0;
    int rc = ws_download_range(ctx, db->ws, 0, db->ws.B, results, m12_pt, m12_ls, inlier_pt, inlier_ls, ctx->s_main);
    if (rc) return rc;
    CK(ctx, cudaStreamSynchronize(ctx->s_main));
    return 0;
}

void plstvo_batch_free(PlContext* ctx, PlDeviceBatch* db) {
    if (!db) return;
    if (ctx) {
        cudaSetDevice(ctx->device);
        cudaDeviceSynchronize();
    }
    db->ws.release();
    delete db;
}

int plstvo_debug_select(PlContext* ctx, int n_lists, const int32_t* off, const double* values, const int32_t* k,
                        const double* pivot, int mode, double* out) {
    if (!ctx || n_lists < 0 || !off || !k || !out || (mode != 0 && mode != 1) || (mode == 1 && !pivot)) return PLSTVO_E_INVALID;
    LOCK(ctx);
    if (n_lists == 0) return 0;
    const size_t n = (size_t)off[n_lists];
    if (n > 0 && !values) return PLSTVO_E_INVALID;
    for (int p = 0; p < n_lists; ++p) {
        const int len = off[p + 1] - off[p];
        if (len < 0 || (len > 0 && (k[p] < 0 || k[p] >= len))) return PLSTVO_E_INVALID;
    }
    CK(ctx, cudaSetDevice(ctx->device));
    const size_t b_v = (n + 2) * 8, b_o = ((size_t)n_lists + 2) * 4, b_k = (size_t)n_lists * 4 + 8, b_p = (size_t)n_lists * 8;
    CK(ctx, ctx->scratch.ensure(b_v + b_o + b_k + 2 * b_p + 64));
    uint8_t* d = ctx->scratch.as<uint8_t>();
    double* dv = reinterpret_cast<double*>(d);
    double* dp = reinterpret_cast<double*>(d + b_v);
    double* dout = reinterpret_cast<double*>(d + b_v + b_p);
    int32_t* doff = reinterpret_cast<int32_t*>(d + b_v + 2 * b_p);
    int32_t* dk = reinterpret_cast<int32_t*>(d + b_v + 2 * b_p + (b_o + 7) / 8 * 8);
    cudaStream_t s = ctx->s_main;
    if (n) CK(ctx, cudaMemcpyAsync(dv, values, n * 8, cudaMemcpyHostToDevice, s));
    CK(ctx, cudaMemcpyAsync(doff, off, ((size_t)n_lists + 1) * 4, cudaMemcpyHostToDevice, s));
    CK(ctx, cudaMemcpyAsync(dk, k, (size_t)n_lists * 4, cudaMemcpyHostToDevice, s));
    if (pivot) CK(ctx, cudaMemcpyAsync(dp, pivot, b_p, cudaMemcpyHostToDevice, s));
    CK(ctx, cudaMemsetAsync(dout, 0, b_p, s));
    CK(ctx, launch_select_selftest(dv, doff, dk, pivot ? dp : nullptr, mode, n_lists, dout, s));
    ctx->launches++;
    CK(ctx, cudaMemcpyAsync(out, dout, b_p, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    return 0;
}

int plstvo_debug_algebra(PlContext* ctx, int n, const double* H, const double* g, double* x, double* lad, double* inv,
                         double* eig) {
    if (!ctx || n < 0 || !H || !g || !x || !lad || !inv || !eig) return PLSTVO_E_INVALID;
    LOCK(ctx);
    if (n == 0) return 0;
    CK(ctx, cudaSetDevice(ctx->device));
    const size_t in_b = (size_t)n * 42 * 8, out_b = (size_t)n * 49 * 8;
    CK(ctx, ctx->scratch.ensure(in_b + out_b));
    double* d = ctx->scratch.as<double>();
    double *dH = d, *dg = d + (size_t)n * 36, *dx = dg + (size_t)n * 6, *dl = dx + (size_t)n * 6, *di = dl + n,
           *de = di + (size_t)n * 36;
    cudaStream_t s = ctx->s_main;
    CK(ctx, cudaMemcpyAsync(dH, H, (size_t)n * 36 * 8, cudaMemcpyHostToDevice, s));
    CK(ctx, cudaMemcpyAsync(dg, g, (size_t)n * 6 * 8, cudaMemcpyHostToDevice, s));
    CK(ctx, launch_algebra_selftest(dH, dg, n, dx, dl, di, de, s));
    ctx->launches++;
    CK(ctx, cudaMemcpyAsync(x, dx, (size_t)n * 6 * 8, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaMemcpyAsync(lad, dl, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaMemcpyAsync(inv, di, (size_t)n * 36 * 8, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaMemcpyAsync(eig, de, (size_t)n * 6 * 8, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    return 0;
}

int plstvo_popc_rate(PlContext* ctx, double* popc_per_s) {
    if (!ctx || !popc_per_s) return PLSTVO_E_INVALID;
    LOCK(ctx);
    CK(ctx, cudaSetDevice(ctx->device));
    const int blocks = ctx->sm_count * 8, iters = 20000;
    CK(ctx, ctx->scratch.ensure((size_t)blocks * 256 * 4));
    cudaEvent_t e0, e1;
    CK(ctx, cudaEventCreate(&e0));
    CK(ctx, cudaEventCreate(&e1));
    CK(ctx, launch_popc_bench(ctx->scratch.as<uint32_t>(), 2000, blocks, ctx->s_main));   // warm-up
    CK(ctx, cudaEventRecord(e0, ctx->s_main));
    CK(ctx, launch_popc_bench(ctx->scratch.as<uint32_t>(), iters, blocks, ctx->s_main));
    CK(ctx, cudaEventRecord(e1, ctx->s_main));
    CK(ctx, cudaEventSynchronize(e1));
    ctx->launches += 2;
    float ms = 0.f;
    CK(ctx, cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *popc_per_s = (double)blocks * 256.0 * iters * 8.0 / (ms * 1e-3);
    return 0;
}

int plstvo_gn_eval_stream(PlContext* ctx, const PlCamera* cam, const PlConfig* cfg, const PlMatchedBatch* m,
                          const double* DT, int iters, double* H, double* g, double* e, float* ms_total) {
    if (!ctx || !cam || !cfg || !m || !DT || iters <= 0) return PLSTVO_E_INVALID;
    LOCK(ctx);
    const int B = m->B;
    if (B <= 0) return 0;
    CK(ctx, cudaSetDevice(ctx->device));
    const size_t n = m->pt_off[B], l = m->ls_off[B];
    cudaStream_t s = ctx->s_main;
    struct Up { const void* src; size_t bytes; };
    const Up ups[8 + 5] = {{m->pt_off, (size_t)(B + 1) * 4}, {m->ls_off, (size_t)(B + 1) * 4}, {m->pt_P, n * 24},
                           {m->pt_pl_obs, n * 16}, {m->pt_sigma2, n * 8}, {m->ls_sP, l * 24}, {m->ls_eP, l * 24},
                           {m->ls_le_obs, l * 24}, {m->ls_spl, l * 16}, {m->ls_epl, l * 16}, {m->ls_sigma2, l * 8},
                           {m->pt_inlier, n}, {m->ls_inlier, l}};
    DevBuf* bufs = ctx->gs_in;   // resident inputs of the roofline run (context lifetime)
    for (int i = 0; i < 13; ++i) {
        CK(ctx, bufs[i].ensure(std::max<size_t>(ups[i].bytes, 16)));
        if (ups[i].src && ups[i].bytes)
            CK(ctx, cudaMemcpyAsync(bufs[i].p, ups[i].src, ups[i].bytes, cudaMemcpyHostToDevice, s));
    }
    MatchedDev md{bufs[0].as<int32_t>(), bufs[1].as<int32_t>(), bufs[2].as<double>(), bufs[3].as<double>(),
                  bufs[4].as<double>(), m->pt_inlier ? bufs[11].as<uint8_t>() : nullptr, bufs[5].as<double>(),
                  bufs[6].as<double>(), bufs[7].as<double>(), bufs[8].as<double>(), bufs[9].as<double>(),
                  bufs[10].as<double>(), m->ls_inlier ? bufs[12].as<uint8_t>() : nullptr};
    // fp32-packed records (SURVEY 8(a) A4/A5: 32 B per point, 64 B per line), packed once on the device
    DevBuf &rec_pt = ctx->gs_rec_pt, &rec_ls = ctx->gs_rec_ls;
    CK(ctx, rec_pt.ensure(std::max<size_t>(n * 32, 32)));
    CK(ctx, rec_ls.ensure(std::max<size_t>(l * 64, 64)));
    CK(ctx, launch_pack_records(md, *cam, B, (int)n, (int)l, rec_pt.as<float4>(), rec_ls.as<float4>(), s));
    ctx->launches++;
    // slices per problem: a work item is ~12 tiles of 16 KB (more slices only when the batch cannot fill the persistent grid)
    int max_tiles = 1;
    for (int p = 0; p < B; ++p)
        max_tiles = std::max(max_tiles, gn_stream_tiles(m->pt_off[p + 1] - m->pt_off[p], m->ls_off[p + 1] - m->ls_off[p]));
    int bpp = std::max(1, std::min(64, max_tiles / 12));
    while ((long)B * bpp < 4L * ctx->sm_count && 2 * bpp <= max_tiles && bpp < 64) ++bpp;
    CK(ctx, ctx->gn_in[0].ensure((size_t)B * 16 * 8));
    CK(ctx, ctx->gn_in[1].ensure((size_t)B * bpp * gn_stream_partials_per_slice() * (ACC_N + 1) * 8));
    CK(ctx, ctx->gn_out[2].ensure((size_t)B * 36 * 8));
    CK(ctx, ctx->gn_out[3].ensure((size_t)B * 7 * 8));
    CK(ctx, cudaMemcpyAsync(ctx->gn_in[0].p, DT, (size_t)B * 16 * 8, cudaMemcpyHostToDevice, s));
    double* dH = ctx->gn_out[2].as<double>();
    double* dg = ctx->gn_out[3].as<double>();
    double* de = dg + (size_t)B * 6;
    cudaEvent_t e0, e1;
    CK(ctx, cudaEventCreate(&e0));
    CK(ctx, cudaEventCreate(&e1));
    auto sweep = [&]() {
        return launch_gn_eval_stream(*cam, *cfg, bufs[0].as<int32_t>(), bufs[1].as<int32_t>(), rec_pt.as<float4>(),
                                     rec_ls.as<float4>(), B, ctx->gn_in[0].as<double>(), ctx->gn_in[1].as<double>(), bpp,
                                     ctx->sm_count, dH, dg, de, s);
    };
    CK(ctx, sweep());   // warm-up
    CK(ctx, cudaEventRecord(e0, s));
    for (int i = 0; i < iters; ++i) CK(ctx, sweep());
    CK(ctx, cudaEventRecord(e1, s));
    ctx->launches += 2 * (iters + 1);
    if (H) CK(ctx, cudaMemcpyAsync(H, dH, (size_t)B * 36 * 8, cudaMemcpyDeviceToHost, s));
    if (g) CK(ctx, cudaMemcpyAsync(g, dg, (size_t)B * 6 * 8, cudaMemcpyDeviceToHost, s));
    if (e) CK(ctx, cudaMemcpyAsync(e, de, (size_t)B * 8, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    float ms = 0.f;
    CK(ctx, cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (ms_total) *ms_total = ms;
    return 0;
}

}  // extern "C"
