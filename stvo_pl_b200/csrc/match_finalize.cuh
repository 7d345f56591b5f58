// match_finalize.cuh — ratio test and mutual filter on K1's merged partials; shared by the standalone
// finalize kernel (match.cu) and the fused per-pair kernel K2 (solve.cu).
#pragma once
#include "common.cuh"

namespace plstvo {

// ---- ratio test + mutual filter ----------------------------------------------------------------------
// (src/matching.cpp:50-61 and :76-86)
__device__ __forceinline__ bool ratio_accept(uint32_t a, uint32_t b, float nnr) {
    // matches_[idx][0].distance < matches_[idx][1].distance * nnr, all float (src/matching.cpp:54);
    // no second neighbour (n2 < 2: UB in the reference) -> no match
    return b != KEY_NONE && (float)(a >> 16) < __fmul_rn((float)(b >> 16), nnr);
}

// m21: 16-bit entries (an index is < 65535 = PLSTVO_MAX_FEATURES; 0xFFFF = no match), so that the largest admissible frame
// (65535 rows: 128 KB) still fits the shared memory of one CTA.
// Unresolved column keys: the tensor-core matcher (match_tc.cu: tc_resolve_kernel) does not recover WHICH query is a train's
// nearest one when that neighbour is unique — the mutual filter does not need the index: query q, whose nearest train is t at
// distance d, is t's unique nearest query exactly when t's best distance equals d.  Such a key carries KEY_IDX_UNRESOLVED
// in its index field, and m21[t] holds M21_DIST | distance instead of an index.  Only used for n1 <= M21_DIST (so that no real
// index collides with the encodings); larger frames get real indices.
constexpr uint16_t M21_NONE = 0xFFFFu;
constexpr uint32_t KEY_IDX_UNRESOLVED = 0xFFFDu;
constexpr uint32_t M21_DIST = 0xFE00u;
__device__ __forceinline__ uint16_t m21_entry(uint32_t key, bool dist_form) {
    const uint32_t idx = key & 0xFFFFu;
    return (uint16_t)((dist_form && idx == KEY_IDX_UNRESOLVED) ? (M21_DIST | (key >> 16)) : idx);
}
__device__ __forceinline__ bool m21_is_mutual(uint16_t e, int q, uint32_t row_key, bool dist_form) {
    if (dist_form && e >= M21_DIST && e != M21_NONE) return (uint32_t)(e & 0x1FFu) == (row_key >> 16);
    return (int)e == q;
}

__device__ __forceinline__ int match_finalize_block(const MatchProblem& pr, uint16_t* m21 /* shared, >= n2 */) {
    const int tid = threadIdx.x, nth = blockDim.x;
    int count = 0;
    if (!pr.enabled) {
        for (int q = tid; q < pr.n1; q += nth) pr.m12[q] = -1;
        return 0;
    }
    const bool dist_form = pr.n1 <= (int)M21_DIST;
    // one partial per row / column: plain streaming loops, unrolled so that several of their independent loads are in
    // flight per thread
#pragma unroll 4
    for (int t = tid; t < pr.n2; t += nth) {
        const uint2 c = pr.colpart[t];
        m21[t] = ratio_accept(c.x, c.y, pr.nnr) ? m21_entry(c.x, dist_form) : M21_NONE;
    }
    __syncthreads();
#pragma unroll 4
    for (int q = tid; q < pr.n1; q += nth) {
        const uint2 c = pr.rowpart[q];
        int32_t i2 = ratio_accept(c.x, c.y, pr.nnr) ? (int32_t)(c.x & 0xFFFFu) : -1;
        if (pr.best_lr && i2 >= 0 && !m21_is_mutual(m21[i2], q, c.x, dist_form)) i2 = -1;
        pr.m12[q] = i2;
        count += (i2 >= 0);
    }
    return count;
}

}  // namespace plstvo
