// match_tc.cu — K1 on the 5th-generation tensor cores: all-pairs 256-bit Hamming 2-NN as a +-1 contraction.
//
// Replaces the arithmetic of StVO::matchNNR / StVO::match (src/matching.cpp:41-91), i.e. OpenCV's
// cv::BFMatcher(NORM_HAMMING)::knnMatch(desc1, desc2, ., 2) per direction.  With descriptor bits mapped to +-1,
//     a . b = (#equal bits) - (#different bits) = 256 - 2 d(a, b)          (exact, |a . b| <= 256)
// so the N1 x N2 distance matrix of one matching problem is a 256-deep GEMM.  Three kernels:
//   tc_expand_kernel   32-byte descriptor rows -> 256 e4m3 bytes (+1.0 = 0x38, -1.0 = 0xB8), written directly in the
//                      128-byte-swizzled K-major operand layout tcgen05.mma reads (tiles of 128 rows = 32 KB contiguous),
//                      so the tiles move with plain bulk copies (UBLKCP) and need no tensor map;
//   tc_hamming_kernel  persistent, warp-specialised: producer warp (bulk copies + mbarriers), one MMA-issuing thread
//                      (tcgen05.mma kind::f8f6f4, 128 x 128 x 32 per instruction, f16 accumulators in TMEM: every partial
//                      sum is an integer of magnitude <= 256, exact in f16), eight epilogue warps reading TMEM with
//                      tcgen05.ld ... .pack::16b: two columns per register.  The hot loop folds only MAXIMA:
//                        row direction   (query -> trains): thread = query row; per 16-column group the packed maximum
//                                         of 8 registers (4 three-input max) is the best of two "sets" (the 8 columns of
//                                         one parity), and a running top-2 over set maxima keeps the best set's tag;
//                        column direction (train -> queries): one packed max per register and row tile (each thread's
//                                         best per column), one cross-lane reduction per work item (not per tile).
//                      Keys carry no indices: the best value, the second over the OTHER sets / lanes (an upper bound
//                      of the second distance) and the best set / lane as a tag;
//   tc_resolve_kernel  merges the per-block partials and converts to distances.  Where the ratio test could pass against
//                      the bound, it re-evaluates the tagged set (8 trains) or lane (queries tag + 128 i) with XOR + POPC:
//                      the exact second distance is min(bound, second within the set / lane), and the scan gives the best
//                      neighbour's index (ties resolved to the lowest index as OpenCV does).  It emits packed keys
//                      (dist << 16 | index) whose unsigned order is OpenCV's (distance, index) order, which the ratio test,
//                      the mutual filter and K2 read.
// Integer-exact end to end: the bit-exact parity tests of the matcher are the acceptance test.
#include <cuda_fp16.h>

#include <cstdio>
#include <cstdlib>

#include "common.cuh"
#include "match_finalize.cuh"
#include "match_tc.cuh"

namespace plstvo {

// ---------------------------------------------------------------------------------------------------------------
// expand: bits -> e4m3 +-1 bytes in the swizzled operand layout
// tile (128 rows) = [slab 0..1][row group 0..15][row 0..7][16-byte chunk position 0..7]; slab = 128 K-bytes;
// logical chunk c of row r sits at position c ^ (r & 7)  (the 128B swizzle: address bits [4,7) ^= bits [7,10))
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) tc_expand_kernel(const TcSide* __restrict__ sides) {
    const TcSide s = sides[blockIdx.y];
    const int tile = blockIdx.x;
    if (tile * TC_ROWS >= s.n) return;
    __shared__ uint32_t lut[16];
    if (threadIdx.x < 16) {
        uint32_t w = 0;
        for (int b = 0; b < 4; ++b) w |= ((threadIdx.x >> b) & 1 ? 0x38u : 0xB8u) << (8 * b);
        lut[threadIdx.x] = w;
    }
    __syncthreads();
    uint8_t* dst_tile = s.dst + (size_t)tile * TC_TILE_BYTES;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int u = it * 256 + threadIdx.x;
        const int c = u & 7, slab = (u >> 3) & 1, r = u >> 4;
        const int row = tile * TC_ROWS + r;
        uint4 out = make_uint4(0, 0, 0, 0);   // rows past the end: zeros (their results are masked, never used)
        if (row < s.n) {
            const uint32_t hw = *reinterpret_cast<const uint16_t*>(s.src + (size_t)row * 32 + slab * 16 + c * 2);
            out = make_uint4(lut[hw & 15], lut[(hw >> 4) & 15], lut[(hw >> 8) & 15], lut[hw >> 12]);
        }
        *reinterpret_cast<uint4*>(dst_tile + slab * 16384 + (r >> 3) * 1024 + (r & 7) * 128 + ((c ^ (r & 7)) * 16)) = out;
    }
}

cudaError_t launch_tc_expand(const TcSide* sides, int n_sides, int max_tiles, cudaStream_t stream) {
    if (n_sides <= 0 || max_tiles <= 0) return cudaSuccess;
    tc_expand_kernel<<<dim3(max_tiles, n_sides), 256, 0, stream>>>(sides);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------------
// PTX helpers (tcgen05 / TMEM)
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tc_mma_f8(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
// 32 lanes x 32 columns of f16 accumulators -> 16 registers, two adjacent columns per register (low half = even column)
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.pack::16b.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// packed f16x2 arithmetic on raw 32-bit registers.  max(max(a, b), c) is fused by ptxas into one 3-input VHMNMX.
__device__ __forceinline__ uint32_t hmax2u(uint32_t a, uint32_t b) {
    uint32_t d;
    asm("max.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
    return d;
}
__device__ __forceinline__ uint32_t hmin2u(uint32_t a, uint32_t b) {
    uint32_t d;
    asm("min.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
    return d;
}
__device__ __forceinline__ uint32_t hne2mask(uint32_t a, uint32_t b) {   // 0xFFFF per half where a != b
    uint32_t d;
    asm("set.ne.u32.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
    return d;
}
__device__ __forceinline__ uint32_t hgt2mask(uint32_t a, uint32_t b) {   // 0xFFFF per half where a > b
    uint32_t d;
    asm("set.gt.u32.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
    return d;
}
__device__ __forceinline__ uint32_t hfma2u(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("fma.rn.f16x2 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t swap16(uint32_t a) { return __byte_perm(a, a, 0x1032); }
__device__ __forceinline__ uint32_t sel32(uint32_t mask, uint32_t a, uint32_t b) { return (mask & a) | (~mask & b); }   // one LOP3
__device__ __forceinline__ uint32_t h2u_lo(uint32_t p) {   // low half (an integer-valued f16 >= 0) -> uint32
    uint32_t d;
    asm("{ .reg .b16 lo, hi; mov.b32 {lo, hi}, %1; cvt.rni.u32.f16 %0, lo; }" : "=r"(d) : "r"(p));
    return d;
}
__device__ __forceinline__ uint32_t h2u_hi(uint32_t p) {
    uint32_t d;
    asm("{ .reg .b16 lo, hi; mov.b32 {lo, hi}, %1; cvt.rni.u32.f16 %0, hi; }" : "=r"(d) : "r"(p));
    return d;
}

// "no value" sentinel: -1024, below every dot value (>= -256)
constexpr uint32_t NEG2 = 0xE400E400u;
constexpr uint32_t H2_NEGHALF = 0xB800B800u, H2_128 = 0x58005800u, H2_511 = 0x5FFC5FFCu;
// (best, second) dot values packed (lo, hi) -> distances d = (256 - v) / 2 (exact), "none" (sentinel) -> 511
__device__ __forceinline__ uint32_t dots_to_dist(uint32_t pv) { return hmin2u(hfma2u(pv, H2_NEGHALF, H2_128), H2_511); }

// running top-2 update with one new packed value: 3 min/max
__device__ __forceinline__ void top2_alu(uint32_t& k1, uint32_t& k2, uint32_t v) {
    const uint32_t t = hmin2u(k1, v);
    k1 = hmax2u(k1, v);
    k2 = hmax2u(k2, t);
}
// maximum of 8 packed registers: 4 VHMNMX
__device__ __forceinline__ uint32_t hmax8(const uint32_t* v) {
    const uint32_t a = hmax2u(hmax2u(v[0], v[1]), v[2]), b = hmax2u(hmax2u(v[3], v[4]), v[5]);
    return hmax2u(hmax2u(hmax2u(a, b), v[6]), v[7]);
}

// shared-memory operand descriptor: K-major, 128-byte swizzle, 8-row groups 1024 B apart (SBO), version 1
__device__ __forceinline__ uint64_t tc_desc(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)0x40004040u << 32);
}
// instruction descriptor: D = f16, A = B = e4m3, both K-major, M = 128, N = 256
constexpr uint32_t TC_IDESC = (uint32_t)((256 >> 3) << 17) | (uint32_t)((TC_ROWS >> 4) << 24);

// ---------------------------------------------------------------------------------------------------------------
// the matcher
// ---------------------------------------------------------------------------------------------------------------
constexpr int TC_OFF_X = 0;
constexpr int TC_OFF_Y = TC_XSTAGES * TC_TILE_BYTES;                      // [slab 0..1][256 rows]: 64 KB
constexpr int TC_OFF_SCR = TC_OFF_Y + 2 * TC_TILE_BYTES;                  // per epilogue warp: 16 x 33 words
constexpr int TC_SCR_WARP = 16 * 33 * 4;
constexpr int TC_OFF_MRG = TC_OFF_SCR + TC_EW * TC_SCR_WARP;              // [groups][4 quarters][columns per group] uint2: 8 KB
constexpr int TC_OFF_BAR = TC_OFF_MRG + 4 * 256 * 8;
constexpr int TC_IRING = 4;                                               // work items announced ahead
constexpr int TC_NBARS = 2 * TC_XSTAGES + 2 + 2 * TC_ASTAGES + 2 * TC_IRING;
constexpr int TC_OFF_RING = TC_OFF_BAR + TC_NBARS * 8;
constexpr int TC_OFF_SLOT = TC_OFF_RING + TC_IRING * 4;
constexpr int TC_SMEM_USED = TC_OFF_SLOT + 16;
static_assert(TC_SMEM_USED + 1024 <= 227 * 1024, "tc_hamming_kernel: shared memory");

size_t tc_smem_bytes() { return (size_t)TC_SMEM_USED + 1024; }

#ifndef TC_MAXNREG
#define TC_MAXNREG 0
#endif
#if TC_MAXNREG > 0
__global__ void __maxnreg__(TC_MAXNREG)
#else
__global__ void __launch_bounds__(TC_THREADS, 1)
#endif
tc_hamming_kernel(const TcProblem* __restrict__ problems, const TcItem* __restrict__ items_a, int n_a,
                  const TcItem* __restrict__ items_b, int n_b, int* __restrict__ sched, __half* __restrict__ debug_tile) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t sbase = (raw + 1023u) & ~1023u;
    uint8_t* sm = smem_raw + (sbase - raw);
    uint64_t* bars = reinterpret_cast<uint64_t*>(sm + TC_OFF_BAR);
    uint64_t* x_full = bars;
    uint64_t* x_empty = bars + TC_XSTAGES;
    uint64_t* y_full = bars + 2 * TC_XSTAGES;
    uint64_t* y_empty = y_full + 1;
    uint64_t* t_full = y_empty + 1;
    uint64_t* t_empty = t_full + TC_ASTAGES;
    uint64_t* i_full = t_empty + TC_ASTAGES;
    uint64_t* i_empty = i_full + TC_IRING;
    volatile int* iring = reinterpret_cast<volatile int*>(sm + TC_OFF_RING);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + TC_OFF_SLOT);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_items = n_a + n_b;

    if (tid == 0) {
        for (int i = 0; i < TC_XSTAGES; ++i) {
            mbar_init(&x_full[i], 1);
            mbar_init(&x_empty[i], 1);
        }
        mbar_init(y_full, 1);
        mbar_init(y_empty, 1);
        for (int i = 0; i < TC_ASTAGES; ++i) {
            mbar_init(&t_full[i], 1);
            mbar_init(&t_empty[i], TC_EW);
        }
        for (int i = 0; i < TC_IRING; ++i) {
            mbar_init(&i_full[i], 1);
            mbar_init(&i_empty[i], TC_EW + 1);   // the MMA thread + the epilogue warps
        }
        fence_mbar_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "n"(TC_ASTAGES * 256)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // work items are handed out by an atomic counter (long ones first: list a, then list b) and announced to the other
    // roles through a small ring in shared memory; -1 ends the kernel
    auto item_at = [&](int it) -> TcItem { return it < n_a ? items_a[it] : items_b[it - n_a]; };

    if (warp == 0) {
        // ===== producer: work distribution + bulk copies of operand tiles =====
        if (lane == 0) {
            uint32_t xs = 0, xph = 0;
            for (uint32_t k = 0;; ++k) {
                const uint32_t slot = k % TC_IRING;
                mbar_wait(&i_empty[slot], ((k / TC_IRING) & 1) ^ 1);
                int it = atomicAdd(sched, 1);
                if (it >= n_items) it = -1;
                iring[slot] = it;
                mbar_arrive(&i_full[slot]);
                if (it < 0) break;
                const TcItem item = item_at(it);
                const TcProblem pr = problems[item.problem];
                const int nyt = (pr.n2 + TC_ROWS - 1) / TC_ROWS, nxt = (pr.n1 + TC_ROWS - 1) / TC_ROWS;
                const int ytiles = min(2, nyt - 2 * item.yblk);
                mbar_wait(y_empty, (k & 1) ^ 1);
                mbar_arrive_expect_tx(y_full, (uint32_t)ytiles * TC_TILE_BYTES);
                for (int h = 0; h < ytiles; ++h)
                    for (int sl = 0; sl < 2; ++sl)
                        bulk_g2s(sm + TC_OFF_Y + sl * 32768 + h * 16384,
                                 pr.ye + (size_t)(2 * item.yblk + h) * TC_TILE_BYTES + sl * 16384, 16384, y_full);
                for (int t = 0; t < nxt; ++t) {
                    mbar_wait(&x_empty[xs], xph ^ 1);
                    mbar_arrive_expect_tx(&x_full[xs], TC_TILE_BYTES);
                    bulk_g2s(sm + TC_OFF_X + xs * TC_TILE_BYTES, pr.xe + (size_t)t * TC_TILE_BYTES, TC_TILE_BYTES,
                             &x_full[xs]);
                    if (++xs == TC_XSTAGES) { xs = 0; xph ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: one thread =====
        if (lane == 0) {
            uint32_t xs = 0, xph = 0, as = 0, aph = 0;
            for (uint32_t k = 0;; ++k) {
                const uint32_t slot = k % TC_IRING;
                mbar_wait(&i_full[slot], (k / TC_IRING) & 1);
                const int it = iring[slot];
                mbar_arrive(&i_empty[slot]);
                if (it < 0) break;
                const TcItem item = item_at(it);
                const TcProblem pr = problems[item.problem];
                const int nxt = (pr.n1 + TC_ROWS - 1) / TC_ROWS;
                mbar_wait(y_full, k & 1);
                for (int t = 0; t < nxt; ++t) {
                    mbar_wait(&t_empty[as], aph ^ 1);
                    mbar_wait(&x_full[xs], xph);
                    tc_fence_after();
                    const uint32_t xa = sbase + TC_OFF_X + xs * TC_TILE_BYTES, ya = sbase + TC_OFF_Y;
                    const uint32_t d = tmem_base + as * 256;
#pragma unroll
                    for (int kk = 0; kk < 8; ++kk)
                        tc_mma_f8(d, tc_desc(xa + (kk >> 2) * 16384 + (kk & 3) * 32),
                                  tc_desc(ya + (kk >> 2) * 32768 + (kk & 3) * 32), TC_IDESC, kk > 0);
                    tc_commit(&x_empty[xs]);
                    tc_commit(&t_full[as]);
                    if (++xs == TC_XSTAGES) { xs = 0; xph ^= 1; }
                    if (++as == TC_ASTAGES) { as = 0; aph ^= 1; }
                }
                tc_commit(y_empty);
            }
        }
    } else {
        // ===== epilogue: TC_EW warps.  quarter q = TMEM lanes 32q..32q+31 (hardware: warp id % 4), group gq = which TC_CW columns
        // of the 256-column accumulator (TC_EW = 8: two groups of 128, two warps per scheduler; TC_EW = 16: four groups of 64, four
        // warps per scheduler: the min / max chains of one warp issue into the dependency stalls of the others)
        constexpr int CW = TC_CW, NCH = CW / 32, NREG = CW / 2;
        const int ew = warp - 2, q = warp & 3, gq = ew >> 2;
        uint32_t* scr = reinterpret_cast<uint32_t*>(sm + TC_OFF_SCR + ew * TC_SCR_WARP);
        uint2* mrg = reinterpret_cast<uint2*>(sm + TC_OFF_MRG) + gq * 4 * CW;
        uint32_t as = 0, aph = 0;
        for (uint32_t k = 0;; ++k) {
            const uint32_t slot = k % TC_IRING;
            mbar_wait(&i_full[slot], (k / TC_IRING) & 1);
            const int it = iring[slot];
            __syncwarp();
            if (lane == 0) mbar_arrive(&i_empty[slot]);
            if (it < 0) break;
            const TcItem item = item_at(it);
            const TcProblem pr = problems[item.problem];
            const int nxt = (pr.n1 + TC_ROWS - 1) / TC_ROWS;
            const int blk = item.yblk * (256 / CW) + gq;      // CW-column block index of this group
            const int ycol0 = blk * CW;
            const int nvalid = min(CW, pr.n2 - ycol0);        // <= 0: nothing for this group
            uint32_t c1[NREG];   // column direction: per register and half, the best value this lane has seen
#pragma unroll
            for (int i = 0; i < NREG; ++i) c1[i] = NEG2;

            for (int t = 0; t < nxt; ++t) {
                mbar_wait(&t_full[as], aph);
                tc_fence_after();
                const int x = t * TC_ROWS + q * 32 + lane;
                const bool xvalid = x < pr.n1;
                // row direction: a "set" is the 8 columns of one parity in a 16-column group; each half of a group maximum
                // is one set's maximum.  Two independent chains keep a running top-2 over set maxima and the group the
                // maximum last rose in: A = registers 0..7 (group 2c), B = registers 8..15 (group 2c + 1)
                uint32_t ra1 = NEG2, ra2 = NEG2, rb1 = NEG2, rb2 = NEG2, ta = 0, tb = 0;
                const uint32_t tad = tmem_base + ((uint32_t)(q * 32) << 16) + as * 256 + gq * CW;
                auto fold = [&](const uint32_t (&v)[16], const int c) {
                    const uint32_t olda = ra1, oldb = rb1;
                    top2_alu(ra1, ra2, hmax8(v));
                    top2_alu(rb1, rb2, hmax8(v + 8));
                    ta = sel32(hne2mask(ra1, olda), (uint32_t)((2 * c) * 0x00010001u), ta);
                    tb = sel32(hne2mask(rb1, oldb), (uint32_t)((2 * c + 1) * 0x00010001u), tb);
#pragma unroll
                    for (int i = 0; i < 16; ++i) c1[c * 16 + i] = hmax2u(c1[c * 16 + i], v[i]);
                };
                if (nvalid == CW && (t + 1) * TC_ROWS <= pr.n1 && debug_tile == nullptr) {
                    // full tile of a full block (the common case): no per-chunk branches, the next chunk's TMEM load is in
                    // flight while this one is folded
                    uint32_t va[16], vb[16];
                    tc_ld32(tad, va);
#pragma unroll
                    for (int c = 0; c < NCH; c += 2) {
                        tc_wait_ld();
                        tc_ld32(tad + (c + 1) * 32, vb);
                        fold(va, c);
                        tc_wait_ld();
                        if (c + 2 < NCH) tc_ld32(tad + (c + 2) * 32, va);
                        fold(vb, c + 1);
                    }
                } else {
#pragma unroll
                    for (int c = 0; c < NCH; ++c) {
                        if (c * 32 >= nvalid) continue;           // warp-uniform: no valid column in this chunk
                        uint32_t v[16];
                        tc_ld32(tad + c * 32, v);
                        tc_wait_ld();
                        if (debug_tile && it == 0 && t == 0) {
#pragma unroll
                            for (int i = 0; i < 16; ++i)
                                *reinterpret_cast<uint32_t*>(debug_tile + (size_t)(q * 32 + lane) * 256 + gq * CW + c * 32 + 2 * i) = v[i];
                        }
                        if (c * 32 + 32 > nvalid) {               // the one boundary chunk of a partial block
#pragma unroll
                            for (int i = 0; i < 16; ++i) {
                                const int col = c * 32 + 2 * i;
                                if (col >= nvalid) v[i] = NEG2;
                                else if (col + 1 >= nvalid) v[i] = (v[i] & 0xFFFFu) | (NEG2 & 0xFFFF0000u);
                            }
                        }
                        if (xvalid) fold(v, c);                   // rows past the end (zero operand rows) contribute nothing
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&t_empty[as]);
                if (++as == TC_ASTAGES) { as = 0; aph ^= 1; }
                if (xvalid && nvalid > 0) {
                    // chains, then the even- and odd-column sets; everything packed, the result sits in the low halves:
                    // the best value, the second over the other sets, the best set as group << 1 | parity
                    const uint32_t m1 = hmax2u(ra1, rb1), m2 = hmax2u(hmax2u(hmin2u(ra1, rb1), ra2), rb2);
                    const uint32_t tg = sel32(hgt2mask(rb1, ra1), tb, ta);
                    const uint32_t s1 = swap16(m1), s2 = swap16(m2), st = swap16(tg);
                    const uint32_t f1 = hmax2u(m1, s1), f2 = hmax2u(hmax2u(hmin2u(m1, s1), m2), s2);
                    const uint32_t tag = sel32(hgt2mask(s1, m1), (st << 1) | 1u, tg << 1) & 0xFu;   // group << 1 | parity
                    const uint32_t dd = dots_to_dist(__byte_perm(f1, f2, 0x5410));
                    pr.rowp[(size_t)blk * pr.n1 + x] = h2u_lo(dd) | (h2u_hi(dd) << 9) | (tag << 18);
                }
            }

            // ---- column direction: reduce the lane maxima over the 128 threads of the group ----
            // per warp: transpose 16 registers at a time through shared memory; lane L folds register (L & 15) over
            // source lanes 16 (L >> 4) .. +15, the two halves meet by shuffle; then the four quarters merge per column.
            // The result: the best value, the second over the other lanes, the best lane (query row mod 128)
#pragma unroll
            for (int p = 0; p < NCH; ++p) {
                const int j = lane & 15, hl = lane >> 4;
#pragma unroll
                for (int i = 0; i < 16; ++i) scr[i * 33 + lane] = c1[p * 16 + i];
                __syncwarp();
                uint32_t m1 = NEG2, m2 = NEG2, id = 0;
#pragma unroll
                for (int kk = 0; kk < 16; ++kk) {
                    const uint32_t v = scr[j * 33 + hl * 16 + kk];
                    const uint32_t tmin = hmin2u(m1, v);
                    const uint32_t nm = hmax2u(m1, v);
                    m2 = hmax2u(m2, tmin);
                    id = sel32(hne2mask(nm, m1), (uint32_t)((hl * 16 + kk) * 0x00010001u), id);
                    m1 = nm;
                }
                __syncwarp();
                // halves: lanes L and L ^ 16 hold the same register over the other 16 source lanes
                const uint32_t o1 = __shfl_xor_sync(0xFFFFFFFFu, m1, 16), o2 = __shfl_xor_sync(0xFFFFFFFFu, m2, 16),
                               oid = __shfl_xor_sync(0xFFFFFFFFu, id, 16);
                const uint32_t n2v = hmax2u(hmax2u(hmin2u(m1, o1), m2), o2);
                const uint32_t n1v = hmax2u(m1, o1);
                const uint32_t nid = sel32(hgt2mask(o1, m1), oid, id);
                if (hl == 0) {
                    const int col = (p * 16 + j) * 2;
                    mrg[q * CW + col] = make_uint2((n1v & 0xFFFFu) | (n2v << 16), nid & 0xFFFFu);
                    mrg[q * CW + col + 1] = make_uint2((n1v >> 16) | (n2v & 0xFFFF0000u), nid >> 16);
                }
            }
            asm volatile("bar.sync %0, 128;" ::"r"(1 + gq) : "memory");
            if (lane < CW / 4) {   // the group's four warps share its CW columns
                const int col = (ew & 3) * (CW / 4) + lane;
                uint32_t b1 = NEG2, b2 = NEG2, bt = 0;   // only the low halves are meaningful
#pragma unroll
                for (int qq = 0; qq < 4; ++qq) {
                    const uint2 e = mrg[qq * CW + col];
                    const uint32_t a1 = e.x & 0xFFFFu, a2 = e.x >> 16;
                    b2 = hmax2u(hmax2u(hmin2u(b1, a1), b2), a2);
                    bt = sel32(hgt2mask(a1, b1), (uint32_t)qq * 32u + e.y, bt);
                    b1 = hmax2u(b1, a1);
                }
                if (col < nvalid) {
                    const uint32_t dd = dots_to_dist(__byte_perm(b1, b2, 0x5410));
                    pr.colp[ycol0 + col] = h2u_lo(dd) | (h2u_hi(dd) << 9) | ((bt & 0x7Fu) << 18);
                }
            }
            asm volatile("bar.sync %0, 128;" ::"r"(1 + gq) : "memory");
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TC_ASTAGES * 256)
                     : "memory");
    }
    // the last CTA out re-arms the scheduler words for the next launch on this stream
    if (tid == 0) {
        __threadfence();
        if (atomicAdd(sched + 1, 1) == (int)gridDim.x - 1) {
            sched[0] = 0;
            sched[1] = 0;
            __threadfence();
        }
    }
}

cudaError_t launch_tc_hamming(const TcProblem* problems, const TcItem* items_a, int n_a, const TcItem* items_b, int n_b,
                              int* sched, int grid, __half* debug_tile, cudaStream_t stream) {
    const int n_items = n_a + n_b;
    if (n_items <= 0) return cudaSuccess;
    static size_t configured[64] = {};
    const size_t smem = tc_smem_bytes();
    cudaError_t e = ensure_dynamic_smem(reinterpret_cast<const void*>(tc_hamming_kernel), smem, configured);
    if (e != cudaSuccess) return e;
    if (grid > n_items) grid = n_items;
    if (getenv("PLSTVO_TC_DIAG")) {
        cudaFuncAttributes fa;
        int occ = -1;
        cudaFuncGetAttributes(&fa, reinterpret_cast<const void*>(tc_hamming_kernel));
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, tc_hamming_kernel, TC_THREADS, smem);
        fprintf(stderr, "[tc diag] regs %d, maxThreadsPerBlock %d, static smem %zu, local %zu, dynamic smem %zu, occupancy %d\n",
                fa.numRegs, fa.maxThreadsPerBlock, fa.sharedSizeBytes, fa.localSizeBytes, smem, occ);
    }
    tc_hamming_kernel<<<grid, TC_THREADS, smem, stream>>>(problems, items_a, n_a, items_b, n_b, sched, debug_tile);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------------
// resolve: values -> distances, candidate tags -> exact indices, packed keys out
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int hamming256(const uint4& a0, const uint4& a1, const uint8_t* p) {
    const uint4 b0 = __ldg(reinterpret_cast<const uint4*>(p)), b1 = __ldg(reinterpret_cast<const uint4*>(p) + 1);
    return __popc(a0.x ^ b0.x) + __popc(a0.y ^ b0.y) + __popc(a0.z ^ b0.z) + __popc(a0.w ^ b0.w) + __popc(a1.x ^ b1.x) +
           __popc(a1.y ^ b1.y) + __popc(a1.z ^ b1.z) + __popc(a1.w ^ b1.w);
}

// exact (best, second) distance from a over the rows j0, j0 + stride, ... (fewer than count of them, below n) of desc;
// i1 = the lowest of those rows at the best distance
__device__ __forceinline__ void scan_top2(const uint4& a0, const uint4& a1, const uint8_t* desc, int j0, int stride, int count,
                                          int n, int& s1, int& s2, int& i1) {
    s1 = s2 = 512;
    i1 = -1;
    for (int i = 0, j = j0; i < count && j < n; ++i, j += stride) {
        const int h = hamming256(a0, a1, desc + (size_t)j * 32);
        if (h < s1) { s2 = s1; s1 = h; i1 = j; }
        else s2 = min(s2, h);
    }
}
// an accepted tie (nnr > 1) or a best the candidates did not hold: lowest index at distance d among all n rows, as OpenCV
// orders them
__device__ __forceinline__ int first_at(const uint4& a0, const uint4& a1, const uint8_t* desc, int n, int d) {
    for (int j = 0; j < n; ++j)
        if (hamming256(a0, a1, desc + (size_t)j * 32) == d) return j;
    return 0;
}

// The partials carry the best distance and an upper bound of the second: the second over the other candidate sets (rows) or
// lanes (columns).  The exact second is min(bound, second within the best set / lane).  When the ratio test already fails
// against the bound it fails against the exact second too (d2 <= bound), so the bound is written as k2 and nothing is
// re-evaluated; ratio_accept (match_finalize.cuh), the only reader of k2, decides the same.  Otherwise the best set / lane is
// re-evaluated with XOR + POPC, which gives the exact second and the index.
__global__ void __launch_bounds__(256) tc_resolve_kernel(const MatchProblem* __restrict__ mps, const TcProblem* __restrict__ tps) {
    const MatchProblem mp = mps[blockIdx.x];
    if (!mp.enabled) return;
    const TcProblem tp = tps[blockIdx.x];
    const int nyh = (mp.n2 + TC_CW - 1) / TC_CW, nxt = (mp.n1 + TC_ROWS - 1) / TC_ROWS;   // row partials: one per TC_CW-train block
    const int slice = blockIdx.y, nslices = gridDim.y;
    // partial word: best distance (9 bits) | second bound << 9 (511 = none) | candidate tag << 18
    // queries: merge over the TC_CW-train blocks (lowest block wins a tie: its indices are lower)
    for (int x = slice * blockDim.x + threadIdx.x; x < mp.n1; x += nslices * blockDim.x) {
        uint32_t b1 = 511, b2 = 511, btag = 0;
        int bh = 0;
        for (int h = 0; h < nyh; ++h) {
            const uint32_t e = __ldg(&tp.rowp[(size_t)h * mp.n1 + x]);
            const uint32_t a1 = e & 511u, a2 = (e >> 9) & 511u;
            b2 = min(max(b1, a1), min(b2, a2));
            if (a1 < b1) { b1 = a1; bh = h; btag = e >> 18; }
        }
        const int d1 = (int)b1;
        uint32_t k2 = KEY_NONE;
        int idx = 0;
        if (mp.n2 >= 2) {
            int d2 = (int)b2;
            if ((float)d1 < __fmul_rn((float)d2, mp.nnr)) {
                // the tagged set: 8 trains of one parity in one 16-column group
                const uint4 a0 = __ldg(reinterpret_cast<const uint4*>(mp.d1 + (size_t)x * 32)),
                            a1 = __ldg(reinterpret_cast<const uint4*>(mp.d1 + (size_t)x * 32) + 1);
                const int base = bh * TC_CW + (int)((btag >> 1) & 7u) * 16 + (int)(btag & 1u);
                int s1, s2, i1;
                scan_top2(a0, a1, mp.d2, base, 2, 8, mp.n2, s1, s2, i1);
                d2 = min(d2, s2);
                if ((float)d1 < __fmul_rn((float)d2, mp.nnr)) idx = d1 != d2 && s1 == d1 ? i1 : first_at(a0, a1, mp.d2, mp.n2, d1);
            }
            k2 = ((uint32_t)d2 << 16) | 0xFFFEu;
        }
        mp.rowpart[x] = make_uint2(((uint32_t)d1 << 16) | (uint32_t)idx, k2);
    }
    // trains: the best lane's queries are rows tag + 128 i
    for (int y = slice * blockDim.x + threadIdx.x; y < mp.n2; y += nslices * blockDim.x) {
        const uint32_t e = __ldg(&tp.colp[y]);
        const int d1 = (int)(e & 511u);
        uint32_t k2 = KEY_NONE;
        int idx = 0;
        if (mp.n1 >= 2) {
            int d2 = (int)((e >> 9) & 511u);
            if ((float)d1 < __fmul_rn((float)d2, mp.nnr)) {
                const uint4 a0 = __ldg(reinterpret_cast<const uint4*>(mp.d2 + (size_t)y * 32)),
                            a1 = __ldg(reinterpret_cast<const uint4*>(mp.d2 + (size_t)y * 32) + 1);
                int s1, s2, i1;
                scan_top2(a0, a1, mp.d1, (int)((e >> 18) & 127u), TC_ROWS, nxt, mp.n1, s1, s2, i1);
                d2 = min(d2, s2);
                if ((float)d1 < __fmul_rn((float)d2, mp.nnr)) {
                    if (d1 != d2 && s1 == d1)
                        // unique best: up to 65024 rows WHICH query it is does not matter to the mutual filter
                        // (match_finalize.cuh: a query whose nearest train is y at distance d1 is that query)
                        idx = mp.n1 <= (int)M21_DIST ? (int)KEY_IDX_UNRESOLVED : i1;
                    else
                        idx = first_at(a0, a1, mp.d1, mp.n1, d1);
                }
            }
            k2 = ((uint32_t)d2 << 16) | 0xFFFEu;
        }
        mp.colpart[y] = make_uint2(((uint32_t)d1 << 16) | (uint32_t)idx, k2);
    }
}

cudaError_t launch_tc_resolve(const MatchProblem* mps, const TcProblem* tps, int n_problems, int slices, cudaStream_t stream) {
    if (n_problems <= 0) return cudaSuccess;
    tc_resolve_kernel<<<dim3(n_problems, slices > 0 ? slices : 1), 256, 0, stream>>>(mps, tps);
    return cudaGetLastError();
}

}  // namespace plstvo
