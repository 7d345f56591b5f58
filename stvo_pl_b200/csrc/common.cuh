// common.cuh — internal declarations shared by the sm_100a kernels and the C-ABI host code.
// Nothing here is part of the public boundary (include/plstvo.h is).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>

#include "../../include/plstvo.h"

namespace plstvo {

constexpr uint32_t KEY_NONE = 0xFFFFFFFFu;  // "no neighbour": larger than any (dist << 16 | idx) key

// ---- K1 (tensor-core matcher, match_tc.cu) result description --------------------------------------
// One matching problem = StVO::match(desc1, desc2) for one feature type of one frame pair
// (src/matching.cpp:63-91).  K1 leaves one merged key pair per row (top-2 trains of each query) and one per
// column (top-2 queries of each train): both directions of the mutual check from ONE pass over the distances.
struct MatchProblem {
    const uint8_t* d1;     // [n1][32]
    const uint8_t* d2;     // [n2][32]
    int32_t n1, n2;
    int32_t enabled;       // 0: Config::hasPoints()/hasLines() false or an empty side -> all -1, no matching
    uint2*  rowpart;       // [n1]  (k1,k2) packed keys (dist << 16 | train index)
    uint2*  colpart;       // [n2]  (k1,k2) packed keys (dist << 16 | query index)
    int32_t* m12;          // [n1] result (problem-local train index or -1)
    float   nnr;
    int32_t best_lr;
};

// ---- K2 (track_solve) ------------------------------------------------------------------------------
constexpr int K2_THREADS = 512;   // one pair per SM at a time: at a few pairs per SM the per-pair latency is what counts
                                  // (128-thread CTAs x 4 per SM were measured: 3x the latency, same throughput at B = 512)
constexpr int K2_WARPS   = K2_THREADS / 32;
constexpr int ACC_N      = 28;    // 21 (upper triangle of J J^T w) + 6 (J r w) + 1 (r^2 w)

// device copies of the PlFrameBatch arrays (all frames of a batch concatenated)
struct FrameDev {
    const int32_t* pt_off;
    const int32_t* ls_off;
    const uint8_t* pdesc;
    const uint8_t* ldesc;
    const double*  pt_P;
    const double*  pt_pl;
    const double*  pt_sigma2;
    const double*  ls_sP;
    const double*  ls_eP;
    const double*  ls_le;
    const double*  ls_spl;
    const double*  ls_epl;
    const double*  ls_sigma2;
    const int32_t* ls_level;
};

// device copy of PlMatchedBatch (explicit matched lists)
struct MatchedDev {
    const int32_t* pt_off;
    const int32_t* ls_off;
    const double*  pt_P;
    const double*  pt_pl_obs;
    const double*  pt_sigma2;
    const uint8_t* pt_inlier;
    const double*  ls_sP;
    const double*  ls_eP;
    const double*  ls_le_obs;
    const double*  ls_spl;
    const double*  ls_epl;
    const double*  ls_sigma2;
    const uint8_t* ls_inlier;
};

struct SolveParams {
    PlCamera cam;
    PlConfig cfg;
    int32_t  mode;            // 0: track (match partials -> mutual -> gather -> optimizePose); 1: explicit lists
    int32_t  first_pair;      // pair index of blockIdx.x == 0
    FrameDev prev, curr;      // mode 0
    MatchedDev matched;       // mode 1
    const MatchProblem* problems;   // mode 0: [2 * pair + {0: points, 1: lines}]
    const PlPrior* priors;    // may be null
    PlPoseResult*  results;
    uint8_t* inlier_pt;       // mode 0: per prev feature; mode 1: per list entry
    uint8_t* inlier_ls;
    // feature storage: shared memory when it fits, else this global scratch (per CTA slice)
    double*  feat_scratch;
    size_t   feat_scratch_stride;  // doubles per CTA
    int32_t  cap_pt, cap_ls;  // capacity of the SoA arrays (max matched features per pair in this launch)
    int32_t  sort_cap;        // power of two >= max(cap_pt, cap_ls)
    int32_t  feat_in_smem;
    long long* phase_cycles;  // optional [pairs][8] debug timers (PLSTVO_PHASE_DEBUG), else null
    const int32_t* only_if;   // optional [pairs]: the CTA of pair p returns at once unless only_if[p] != 0
};

// ---- streamed optimizePose (solve.cu + gn_stream.cu): frames whose matched lists do not fit K2's shared memory ------------
// GN evaluations run as sweeps of gn_eval_stream_kernel over the fp32-packed records of ALL problems of the launch (HBM-bound),
// a one-warp-per-problem step kernel does the 6x6 solve / pose update / stop tests between sweeps, removeOutliers and the
// finalisation stay double precision on the fp64 lists.  Problems that leave the common path (robust fallback, solver_mode 1)
// are handed to K2 (global-scratch form) through SolveParams::only_if.
struct StreamCtl {            // per problem
    double DT0[16];           // initial pose of optimizePose
    double cov[36];
    double err, err_prev;
    int32_t iters, phase, fail_first, delegate, done, status, iters1, iters2, n_inl_p, n_inl_l, np, nl;
};
struct StreamBufs {
    float4*  rec_pt;          // 2 float4 per point slot, tile-planar (gn_stream.cu)
    float4*  rec_ls;          // 4 float4 per line slot
    int32_t* cnt_pt;          // [B] live records per problem
    int32_t* cnt_ls;
    double*  DT;              // [B][16] pose being optimised: read and updated by the GN loop kernel
    int32_t* active;          // [B]
    StreamCtl* ctl;           // [B]
    uint8_t* flag_pt;         // inlier flags per list entry (slots of the prev frame / of the explicit list)
    uint8_t* flag_ls;
    uint16_t* midx_pt;        // prev index of list entry k (track mode)
    uint16_t* midx_ls;
    int32_t* queue;           // problem queues of the persistent GN kernel (one int per launch of a solve: [2] per chunk)
    int32_t  sm_count;
};
// prm.feat_scratch must hold k2_feat_stride() doubles per pair; prm.feat_in_smem must be 0
cudaError_t launch_stream_solve(const SolveParams& prm, int n_pairs, const StreamBufs& sb, cudaStream_t stream, int* launches,
                                cudaEvent_t* marks = nullptr);   // marks: 4 events (see solve.cu), instrumentation only

size_t k2_smem_bytes(int cap_pt, int cap_ls, int sort_cap, bool feat_in_smem);
size_t k2_feat_stride(int cap_pt, int cap_ls);   // doubles of global feature scratch per pair

// kernel launchers (defined in match.cu / solve.cu)
cudaError_t launch_match_finalize(const MatchProblem* problems, int n_problems, int max_n2, int32_t* counts,
                                  cudaStream_t stream);
cudaError_t launch_track_solve(const SolveParams& prm, int n_pairs, cudaStream_t stream);
cudaError_t launch_select_selftest(const double* v, const int32_t* off, const int32_t* ks, const double* pivot, int mode, int n_lists,
                                   double* out, cudaStream_t stream);
cudaError_t launch_algebra_selftest(const double* H, const double* g, int n, double* x, double* lad, double* inv,
                                    double* eig, cudaStream_t stream);
cudaError_t launch_popc_bench(uint32_t* out, int iters, int blocks, cudaStream_t stream);

// ---- StVO::matchGrid (match_grid.cu) ---------------------------------------------------------------------------
struct GridProblem {          // one frame: queries = left image, trains = right image
    int32_t n1, n2;
    const int32_t* q_cell;    // points: [n1][2]; lines: [n1][4] (sp.x, sp.y, ep.x, ep.y)
    const uint8_t* d1;
    const int32_t* t_cell;    // points: [n2][2]
    const double*  t_line;    // lines: [n2][4] in grid units
    const double*  t_dir;     // lines: [n2][2]
    const uint8_t* d2;
    int32_t* m12;             // [n1]
    int32_t* count;           // matches (or a negative error code)
    // scratch
    int32_t* grid_items;
    int2*    q_pairs;         // [n1][cap] (i2, d)
    int32_t* q_count;         // [n1]
    int32_t* t_count;         // [n2]
    int32_t* t_start;         // [n2 + 1]
    int32_t* t_slots;         // [n1 * cap]
    uint8_t* seen;            // [n1 * cap]
    int32_t* m21;             // [n2]
};
struct GridParams {
    int32_t rows, cols, cap, best_lr;
    PlGridWindow w;
    double ratio, line_sim_th;
};
size_t match_grid_smem_bytes(int rows, int cols);
cudaError_t launch_match_grid(const GridProblem* problems, int B, const GridParams& prm, bool lines, cudaStream_t stream);
// lift.cu: grid coordinates of raw key points / key lines (the loops in front of matchGrid, src/stereoFrame.cpp:129-139, :318-337)
cudaError_t launch_stereo_cells_points(int n_l, int n_r, double inv_w, double inv_h, const float* kp_l, const float* kp_r,
                                       int32_t* q_cell, int32_t* t_cell, cudaStream_t s);
cudaError_t launch_stereo_cells_lines(int n_l, int n_r, double inv_w, double inv_h, const float* seg_l, const float* seg_r,
                                      int32_t* q_line, double* t_line, double* t_dir, cudaStream_t s);
// lift.cu: stereo matches -> PointFeature / LineFeature records (src/stereoFrame.cpp:149-172, :348-397)
cudaError_t launch_lift_points(const PlCamera& cam, const PlStereoConfig& sc, int B, const int32_t* l_off, const float* kp_l,
                               const int32_t* oct_l, const uint8_t* desc_l, const int32_t* r_off, const float* kp_r,
                               const int32_t* m12, double* pt_pl, double* pt_disp, double* pt_P, double* pt_sigma2,
                               int32_t* pt_level, uint8_t* pdesc_out, int32_t* src_idx, int32_t* counts, cudaStream_t s,
                               const int32_t* out_off = nullptr);   // out_off: compact output offsets per frame (else l_off); null outputs are skipped
cudaError_t launch_lift_lines(const PlCamera& cam, const PlStereoConfig& sc, int B, const int32_t* l_off, const float* seg_l,
                              const float* ang_l, const int32_t* oct_l, const uint8_t* desc_l, const int32_t* r_off,
                              const float* seg_r, const int32_t* m12, double* ls_spl, double* ls_epl, double* ls_sdisp,
                              double* ls_edisp, double* ls_sP, double* ls_eP, double* ls_le, double* ls_angle,
                              double* ls_sigma2, int32_t* ls_level, uint8_t* ldesc_out, int32_t* src_idx, int32_t* counts,
                              cudaStream_t s, const int32_t* out_off = nullptr);

// GN evaluation streamed from HBM (roofline kernel of config C5): fp32-packed records, TMA-staged tiles
int gn_stream_tiles(int n_pt, int n_ls);
int gn_stream_partials_per_slice();   // fp64 partial records one slice writes (one per consumer warp)   // 16 KB tiles of one problem (512 points or 256 lines each)
cudaError_t launch_pack_records(const MatchedDev& m, const PlCamera& cam, int B, int n_pt, int n_ls, float4* pt, float4* ls,
                                cudaStream_t stream);
cudaError_t launch_gn_eval_stream(const PlCamera& cam, const PlConfig& cfg, const int32_t* pt_off, const int32_t* ls_off,
                                  const float4* pt, const float4* ls, int B, const double* DT, double* partial,
                                  int slices_per_problem, int sm_count, double* H, double* g, double* e, cudaStream_t stream);

// cudaFuncSetAttribute is per device: a process may drive several GPUs (one context each), so the opted-in dynamic
// shared-memory size is remembered per device (`done`: one slot per device ordinal, zero-initialised by the caller).
inline cudaError_t ensure_dynamic_smem(const void* fn, size_t bytes, size_t* done /* [64] */) {
    static std::mutex mu;   // the caches are per function, contexts (and their locks) are per device: two contexts on one
    std::lock_guard<std::mutex> lock(mu);   // device may launch the same kernel concurrently
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    size_t& have = done[dev & 63];
    if (bytes <= have) return cudaSuccess;
    e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) have = bytes;
    return e;
}

// ---- PTX helpers: mbarrier + 1-D bulk async copy (TMA engine, UBLKCP in SASS) ------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// global -> shared bulk copy completing on an mbarrier; addresses and size must be multiples of 16 B
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(smem_dst)),
        "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

}  // namespace plstvo
