// match_tc.cuh — work description of the tensor-core form of K1 (match_tc.cu).  Internal, not part of the boundary.
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"

namespace plstvo {

constexpr int TC_ROWS = 128;                    // descriptor rows per operand tile (UMMA M and N)
constexpr int TC_TILE_BYTES = TC_ROWS * 256;    // 128 rows x 256 e4m3 bytes, swizzled K-major layout
#ifndef TC_EPILOGUE_WARPS
#define TC_EPILOGUE_WARPS 8
#endif
// epilogue warps: 8 (two per scheduler, 128 accumulator columns each) or 16 (four per scheduler, 64 columns each: 96 registers per
// thread).  Measured on 512 C2 pairs: 8 warps 0.627 ms; 16 warps 0.664 ms, 0.625 ms with half of the column updates moved to the FMA
// pipe (a variant since removed) — no gain, so 8 stays the default and -DTC_EPILOGUE_WARPS=16 remains a build option.
constexpr int TC_EW = TC_EPILOGUE_WARPS;
constexpr int TC_CW = 1024 / TC_EW;             // accumulator columns per epilogue warp = trains per row-partial block
constexpr int TC_XSTAGES = TC_EW == 16 ? 3 : 4; // query tiles in flight (shared memory ring; 16 warps need the room for their scratch)
constexpr int TC_ASTAGES = 2;                   // accumulator stages in TMEM (256 columns each)
constexpr int TC_THREADS = 64 + 32 * TC_EW;     // producer warp + MMA warp + the epilogue warps
static_assert(TC_EW == 8 || TC_EW == 16, "epilogue warps");

// one descriptor matrix to expand (queries or trains of one matching problem)
struct TcSide {
    const uint8_t* src;   // [n][32] descriptor rows
    int32_t n;
    uint8_t* dst;         // ceil(n / 128) tiles of TC_TILE_BYTES
};

// one matching problem = StVO::match(desc1, desc2): queries stream through the M side, trains sit on the N side
struct TcProblem {
    const uint8_t* xe;    // expanded queries  (desc1): ceil(n1 / 128) tiles
    const uint8_t* ye;    // expanded trains   (desc2): ceil(n2 / 128) tiles
    int32_t n1, n2;
    // partials: best distance | second << 9 (511 = none) | tag << 18, where "second" is the second over the other candidate
    // sets (rows) or lanes (columns), an upper bound of the exact second distance that tc_resolve_kernel refines
    uint32_t* rowp;       // [ceil(n2 / TC_CW)][n1]: tag = best set (16-column group << 1 | parity: 8 trains)
    uint32_t* colp;       // [n2]:                 tag = best lane (query row mod 128)
};

// one work item of the persistent kernel: all query tiles of a problem against 256 trains
struct TcItem {
    int32_t problem;
    int32_t yblk;
};

size_t tc_smem_bytes();
cudaError_t launch_tc_expand(const TcSide* sides, int n_sides, int max_tiles, cudaStream_t stream);
// items_a then items_b form the work list (long items first); sched: two zeroed ints per concurrently running launch
cudaError_t launch_tc_hamming(const TcProblem* problems, const TcItem* items_a, int n_a, const TcItem* items_b, int n_b,
                              int* sched, int grid, __half* debug_tile, cudaStream_t stream);
// writes MatchProblem::rowpart[n1] / colpart[n2] as packed keys (dist << 16 | index)
cudaError_t launch_tc_resolve(const MatchProblem* mps, const TcProblem* tps, int n_problems, int slices, cudaStream_t stream);

}  // namespace plstvo
