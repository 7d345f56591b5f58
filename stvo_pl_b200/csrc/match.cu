// match.cu — the standalone match finalize and the POPC issue-rate micro-benchmark (sm_100a).
//
// match_finalize_kernel: one CTA per matching problem runs match_finalize_block (ratio test + mutual filter,
// match_finalize.cuh) on the partials K1 (match_tc.cu) left and counts the matches.  plstvo_match_batch and
// plstvo_f2f_tracking call it; in track mode K2 (solve.cu) runs the same block function itself.
#include "common.cuh"
#include "match_finalize.cuh"

namespace plstvo {

__global__ void __launch_bounds__(256) match_finalize_kernel(const MatchProblem* __restrict__ problems,
                                                             int32_t* __restrict__ counts) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ int s_count;
    if (threadIdx.x == 0) s_count = 0;
    __syncthreads();
    const MatchProblem pr = problems[blockIdx.x];
    int c = match_finalize_block(pr, reinterpret_cast<uint16_t*>(smem));
    for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_count, c);
    __syncthreads();
    if (threadIdx.x == 0 && counts) counts[blockIdx.x] = s_count;
}

cudaError_t launch_match_finalize(const MatchProblem* problems, int n_problems, int max_n2, int32_t* counts,
                                  cudaStream_t stream) {
    if (n_problems <= 0) return cudaSuccess;
    const size_t smem = ((size_t)(max_n2 > 0 ? max_n2 : 1) * sizeof(uint16_t) + 15) / 16 * 16;
    static size_t configured[64] = {};
    if (smem > 48 * 1024) {
        cudaError_t e = ensure_dynamic_smem(reinterpret_cast<const void*>(match_finalize_kernel), smem, configured);
        if (e != cudaSuccess) return e;
    }
    match_finalize_kernel<<<n_problems, 256, smem, stream>>>(problems, counts);
    return cudaGetLastError();
}

// ---- POPC issue-rate micro-benchmark (plstvo_popc_rate) ---------------------------------------------
__global__ void __launch_bounds__(256) popc_bench_kernel(uint32_t* out, int iters) {
    uint32_t x0 = threadIdx.x * 2654435761u + blockIdx.x, x1 = x0 ^ 0x9E3779B9u, x2 = x0 + 0x7F4A7C15u,
             x3 = x1 * 3u, x4 = x0 ^ 0x12345u, x5 = x1 + 77u, x6 = x2 ^ 0xABCDEFu, x7 = x3 + 1234567u;
    uint32_t acc = 0;
    for (int i = 0; i < iters; ++i) {
        // 8 independent POPCs per iteration, inputs perturbed so nothing folds
        acc += __popc(x0) + __popc(x1) + __popc(x2) + __popc(x3) + __popc(x4) + __popc(x5) + __popc(x6) + __popc(x7);
        x0 ^= acc; x1 += x0; x2 ^= x1; x3 += x2; x4 ^= x3; x5 += x4; x6 ^= x5; x7 += x6;
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = acc;
}

cudaError_t launch_popc_bench(uint32_t* out, int iters, int blocks, cudaStream_t stream) {
    popc_bench_kernel<<<blocks, 256, 0, stream>>>(out, iters);
    return cudaGetLastError();
}

}  // namespace plstvo
