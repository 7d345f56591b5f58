// solve.cu — K2: one persistent CTA per frame pair does everything after the distance tiles:
//   A. ratio test and mutual filter on K1's partials         (src/matching.cpp:50-61, :76-86)
//   B. build matched_pt / matched_ls in ascending prev index  (src/stereoFrameHandler.cpp:144-152, :167-179)
//      as structure-of-arrays in shared memory (coalesced, conflict-free), with the per-feature constants of the
//      evaluator (sqrt(sigma2), the line-overlap coefficients) computed once
//   C. optimizePose                                            (src/stereoFrameHandler.cpp:307-392):
//      Gauss-Newton (:394-431) / robust Gauss-Newton (:433-480): all threads evaluate the per-feature residual,
//      1x6 Jacobian row and Cauchy weight (:549-694, :696-962); a transposed warp reduction + one shared-memory
//      pass give the 21 + 6 + 1 normal-equation sums; warp 0 then solves the 6x6 system with lanes-as-columns
//      Householder QR, updates the SE(3) pose and evaluates the stop tests, all on-chip;
//      removeOutliers (:988-1067) with median / MAD (src/auxiliar.cpp:387-430) from a segment-local bitonic sort
//      and a binary search on the V-shaped deviation sequence; isGoodSolution (:292-305) with a parallel-order
//      Jacobi eigen-solver; pose finalisation (:372-391).
// Features are read from HBM exactly once per solve; every GN evaluation runs out of shared memory.
// All arithmetic is double precision like the reference (B200 has a full-rate FP64 pipe).  Summation order,
// reciprocal-multiplies and the 6x6 algorithms differ from the reference at rounding level (1e-16 relative),
// far inside the 1e-5 rad / 1e-4 m bar; the reduction order is fixed, so results are run-to-run deterministic.
#include <math.h>

#include "common.cuh"
#include "gn_stream.cuh"
#include "match_finalize.cuh"

namespace plstvo {

#define FULL_MASK 0xFFFFFFFFu

// ---- SoA views of the matched lists --------------------------------------------------------------
struct Feat {
    double *Px, *Py, *Pz, *pu, *pv, *pss;                                          // points (pss = sqrt(sigma2))
    double *sX, *sY, *sZ, *eX, *eY, *eZ, *l0, *l1, *l2, *oa, *ob, *oc, *lss;       // lines  (oa,ob,oc: overlap)
    uint8_t *inl_p, *inl_l;
    int np, nl;
};
constexpr int PT_ARRAYS = 6, LS_ARRAYS = 13;

struct State {
    double red[K2_WARPS][32];
    double acc[32];          // reduced sums: H upper triangle (21), g (6), e (1), count (1)
    double DT[16];           // pose being optimised
    double DT0[16];          // initial pose of optimizePose
    double H[36];            // normal matrix of the last evaluation (row-major, symmetric)
    double cov[36];
    double err;
    double scal[4];
    double sum[K2_WARPS][4];
    int    ctrl;             // loop control broadcast
    int    n_inl_p, n_inl_l;
    int    evals;
    int    scan[K2_WARPS];
    long long tc[8];         // debug phase timers: 0 match-finalize 1 gather 2 GN-eval 3 GN-serial 4 gates/eig 5 outliers 6 final 7 sort+MAD (inside 5)
    PlPoseResult out;
};

__host__ __device__ inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

size_t k2_smem_bytes(int cap_pt, int cap_ls, int sort_cap, bool feat_in_smem) {
    size_t b = align_up(sizeof(State), 16);
    b += (size_t)sort_cap * sizeof(double);
    b += align_up((size_t)cap_pt, 16) + align_up((size_t)cap_ls, 16);                      // inlier flags
    b += align_up((size_t)cap_pt * 2, 16) + align_up((size_t)cap_ls * 2, 16);              // prev index of entry k
    if (feat_in_smem) b += ((size_t)PT_ARRAYS * cap_pt + (size_t)LS_ARRAYS * cap_ls) * sizeof(double);
    return b;
}

size_t k2_feat_stride(int cap_pt, int cap_ls) { return (size_t)PT_ARRAYS * cap_pt + (size_t)LS_ARRAYS * cap_ls; }

__device__ __forceinline__ double shfl(double v, int src) { return __shfl_sync(FULL_MASK, v, src); }
__device__ __forceinline__ double shfl_xor(double v, int m) { return __shfl_xor_sync(FULL_MASK, v, m); }
__device__ __forceinline__ double sum8(double v) {   // sum over each aligned group of 8 lanes
    v += shfl_xor(v, 1);
    v += shfl_xor(v, 2);
    v += shfl_xor(v, 4);
    return v;
}
__device__ __forceinline__ int tri(int i, int j) { return i * 6 - (i * (i - 1)) / 2 + (j - i); }   // i <= j
__device__ __forceinline__ double sel6(const double* a, int i) {   // a[i] with a register-resident a
    double r = a[0];
#pragma unroll
    for (int k = 1; k < 6; k++) r = (i == k) ? a[k] : r;
    return r;
}
__device__ __forceinline__ double sel9(const double* a, int i) {
    double r = a[0];
#pragma unroll
    for (int k = 1; k < 9; k++) r = (i == k) ? a[k] : r;
    return r;
}

// ---- small SE(3) helpers: every lane of the calling warp computes the same thing in registers -------------
__device__ __forceinline__ void mat4_identity(double* T) {
#pragma unroll
    for (int i = 0; i < 16; i++) T[i] = (i % 5 == 0) ? 1.0 : 0.0;
}
__device__ __forceinline__ void mat4_mul(const double* A, const double* B, double* C) {   // C must not alias A or B
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) {
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < 4; k++) s += A[i * 4 + k] * B[k * 4 + j];
            C[i * 4 + j] = s;
        }
}
__device__ __forceinline__ bool mat4_is_identity(const double* T) {
    bool id = true;
#pragma unroll
    for (int i = 0; i < 16; i++) id = id && (T[i] == ((i % 5 == 0) ? 1.0 : 0.0));
    return id;
}
__device__ __forceinline__ void mat3_mul(const double* A, const double* B, double* C) {
#pragma unroll
    for (int i = 0; i < 3; i++)
#pragma unroll
        for (int j = 0; j < 3; j++) C[i * 3 + j] = A[i * 3] * B[j] + A[i * 3 + 1] * B[3 + j] + A[i * 3 + 2] * B[6 + j];
}
__device__ __forceinline__ void skew3(double x, double y, double z, double* S) {  // src/auxiliar.cpp:29-44
    S[0] = 0;  S[1] = -z; S[2] = y;
    S[3] = z;  S[4] = 0;  S[5] = -x;
    S[6] = -y; S[7] = x;  S[8] = 0;
}
__device__ __forceinline__ void inverse_se3(const double* T, double* Ti) {  // src/auxiliar.cpp:113-122
    mat4_identity(Ti);
#pragma unroll
    for (int i = 0; i < 3; i++) {
        double s = 0.0;
#pragma unroll
        for (int j = 0; j < 3; j++) {
            Ti[i * 4 + j] = T[j * 4 + i];
            s += T[j * 4 + i] * T[j * 4 + 3];
        }
        Ti[i * 4 + 3] = -s;
    }
}
__device__ __forceinline__ void expmap_se3(const double* x, double* T) {  // src/auxiliar.cpp:124-141, x = [t; w]
    double t0 = x[0], t1 = x[1], t2 = x[2];
    double R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    const double theta = sqrt(x[3] * x[3] + x[4] * x[4] + x[5] * x[5]);
    if (!(theta < 0.000001)) {
        double s[9], ss[9], V[9];
        const double it = 1.0 / theta;
        skew3(x[3] * it, x[4] * it, x[5] * it, s);
        mat3_mul(s, s, ss);
        double sn, cs;
        sincos(theta, &sn, &cs);
        const double a = (1.0 - cs) * it, b = (theta - sn) * it;
#pragma unroll
        for (int i = 0; i < 9; i++) {
            const double I = (i % 4 == 0) ? 1.0 : 0.0;
            R[i] = I + s[i] * sn + ss[i] * (1.0 - cs);
            V[i] = I + s[i] * a + ss[i] * b;
        }
        const double u0 = V[0] * t0 + V[1] * t1 + V[2] * t2, u1 = V[3] * t0 + V[4] * t1 + V[5] * t2,
                     u2 = V[6] * t0 + V[7] * t1 + V[8] * t2;
        t0 = u0; t1 = u1; t2 = u2;
    }
    mat4_identity(T);
#pragma unroll
    for (int i = 0; i < 3; i++)
#pragma unroll
        for (int j = 0; j < 3; j++) T[i * 4 + j] = R[i * 3 + j];
    T[3] = t0; T[7] = t1; T[11] = t2;
}
__device__ __forceinline__ void mat3_inverse(const double* A, double* Ai) {
    const double c00 = A[4] * A[8] - A[5] * A[7], c01 = A[5] * A[6] - A[3] * A[8], c02 = A[3] * A[7] - A[4] * A[6];
    const double id = 1.0 / (A[0] * c00 + A[1] * c01 + A[2] * c02);
    Ai[0] = c00 * id; Ai[1] = (A[2] * A[7] - A[1] * A[8]) * id; Ai[2] = (A[1] * A[5] - A[2] * A[4]) * id;
    Ai[3] = c01 * id; Ai[4] = (A[0] * A[8] - A[2] * A[6]) * id; Ai[5] = (A[2] * A[3] - A[0] * A[5]) * id;
    Ai[6] = c02 * id; Ai[7] = (A[1] * A[6] - A[0] * A[7]) * id; Ai[8] = (A[0] * A[4] - A[1] * A[3]) * id;
}
__device__ __forceinline__ void logmap_se3(const double* T, double* x) {  // src/auxiliar.cpp:143-173
    double V[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, w0 = 0, w1 = 0, w2 = 0;
    double cosine = (T[0] + T[5] + T[10] - 1.0) / 2.0;
    if (cosine > 1.0) cosine = 1.0;
    else if (cosine < -1.0) cosine = -1.0;
    double sine = sqrt(1.0 - cosine * cosine);
    if (sine > 1.0) sine = 1.0;
    const double theta = acos(cosine);
    if (theta > 0.000001) {
        const double f = theta / (2.0 * sine);
        w0 = f * (T[9] - T[6]);      // skewcoords(theta (R - R^T) / (2 sine)): M(2,1), M(0,2), M(1,0)
        w1 = f * (T[2] - T[8]);
        w2 = f * (T[4] - T[1]);
        double s[9], ss[9];
        const double it = 1.0 / theta;
        skew3(w0 * it, w1 * it, w2 * it, s);
        mat3_mul(s, s, ss);
        const double a = (1.0 - cosine) * it, b = (theta - sine) * it;
#pragma unroll
        for (int i = 0; i < 9; i++) V[i] = ((i % 4 == 0) ? 1.0 : 0.0) + s[i] * a + ss[i] * b;
    }
    double Vi[9];
    mat3_inverse(V, Vi);
    x[0] = Vi[0] * T[3] + Vi[1] * T[7] + Vi[2] * T[11];
    x[1] = Vi[3] * T[3] + Vi[4] * T[7] + Vi[5] * T[11];
    x[2] = Vi[6] * T[3] + Vi[7] * T[7] + Vi[8] * T[11];
    x[3] = w0; x[4] = w1; x[5] = w2;
}

// ---- 6x6 algebra on ONE warp, lane j holding column j -----------------------------------------------------
// ColPivHouseholderQR<Matrix6d>(H).solve(g) and logAbsDeterminant (src/stereoFrameHandler.cpp:417-418, :453-455).
// Lanes 0..5 hold the columns of H, lane 6 the right-hand side.  Every lane returns x[6] and log|det|.
template <bool NEED_LAD>
__device__ void warp_qr6_solve(const double* Hs /* shared, row-major symmetric */, const double* gs, double* x,
                               double& log_abs_det) {
    const int lane = threadIdx.x & 31;
    double a[6];
#pragma unroll
    for (int i = 0; i < 6; i++) a[i] = (lane < 6) ? Hs[i * 6 + lane] : (lane == 6 ? gs[i] : 0.0);
    int pj = lane;
    double maxpivot = 0.0;
#pragma unroll
    for (int k = 0; k < 6; k++) {
        double nrm = 0.0;
#pragma unroll
        for (int i = k; i < 6; i++) nrm += a[i] * a[i];
        if (lane < k || lane > 5) nrm = -1.0;
        double bv = nrm;
        int bl = lane;
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) {   // first maximum over lanes 0..7 (lowest lane on ties, like Eigen's maxCoeff)
            const double ov = shfl_xor(bv, o);
            const int ol = __shfl_xor_sync(FULL_MASK, bl, o);
            if (ov > bv || (ov == bv && ol < bl)) { bv = ov; bl = ol; }
        }
        bl = __shfl_sync(FULL_MASK, bl, 0);
        const int src = (lane == k) ? bl : ((lane == bl) ? k : lane);   // swap columns k <-> bl
#pragma unroll
        for (int i = 0; i < 6; i++) a[i] = shfl(a[i], src);
        pj = __shfl_sync(FULL_MASK, pj, src);
        double ck[6], v[6];
#pragma unroll
        for (int i = 0; i < 6; i++) ck[i] = (i >= k) ? shfl(a[i], k) : 0.0;
        double tail = 0.0;
#pragma unroll
        for (int i = k + 1; i < 6; i++) tail += ck[i] * ck[i];
        const double c0 = ck[k];
        double beta, tau;
        if (tail <= 2.2250738585072014e-308) {
            tau = 0.0;
            beta = c0;
#pragma unroll
            for (int i = 0; i < 6; i++) v[i] = 0.0;
        } else {
            beta = sqrt(c0 * c0 + tail);
            if (c0 >= 0.0) beta = -beta;
            const double iden = 1.0 / (c0 - beta);
#pragma unroll
            for (int i = 0; i < 6; i++) v[i] = (i > k) ? ck[i] * iden : 0.0;
            tau = (beta - c0) / beta;
        }
        v[k] = 1.0;
        if (lane > k && lane <= 6) {
            double s = 0.0;
#pragma unroll
            for (int i = k; i < 6; i++) s += v[i] * a[i];
            s *= tau;
#pragma unroll
            for (int i = k; i < 6; i++) a[i] -= s * v[i];
        }
        if (lane == k) {
#pragma unroll
            for (int i = k; i < 6; i++) a[i] = (i == k) ? beta : 0.0;
        }
        maxpivot = fmax(maxpivot, fabs(beta));
    }
    double d[6], c[6], y[6];
    int perm[6];
#pragma unroll
    for (int k = 0; k < 6; k++) {
        d[k] = shfl(a[k], k);
        c[k] = shfl(a[k], 6);
        perm[k] = __shfl_sync(FULL_MASK, pj, k);
    }
    const double thr = maxpivot * (2.220446049250313e-16 * 6.0);
    int rank = 0;
    double lad = 0.0, rd[6];
#pragma unroll
    for (int k = 0; k < 6; k++) {
        rank += (fabs(d[k]) > thr) ? 1 : 0;
        if (NEED_LAD) lad += log(fabs(d[k]));
        rd[k] = 1.0 / d[k];             // six independent reciprocals: pipelined, off the substitution's chain
    }
    log_abs_det = lad;
#pragma unroll
    for (int k = 5; k >= 0; k--) {
        double s = c[k];
#pragma unroll
        for (int j = k + 1; j < 6; j++) {
            const double rkj = shfl(a[k], j);
            if (j < rank) s -= rkj * y[j];
        }
        y[k] = (k < rank) ? s * rd[k] : 0.0;
    }
#pragma unroll
    for (int i = 0; i < 6; i++) {
        double xi = 0.0;
#pragma unroll
        for (int k = 0; k < 6; k++) xi = (perm[k] == i) ? y[k] : xi;
        x[i] = xi;
    }
}

// Fast path of the solve: H is symmetric positive definite whenever the problem is well posed, so a lanes-as-columns
// Cholesky (6 rsqrt on the critical path instead of the QR's pivot searches, square roots and divisions) gives the
// same x to rounding.  Returns false — and the caller runs the column-pivoted QR, which also handles rank deficiency
// like Eigen — when a pivot is not safely positive.
// `lad` (optional): log|det H| = sum of the logs of the Cholesky pivots, what the robust loop tests the sign of (:455-459).
__device__ bool warp_chol6_solve(const double* Hs, const double* gs, double* x, double* lad = nullptr) {
    const int lane = threadIdx.x & 31;
    const int lj = (lane < 6) ? lane : 0;
    double a[6];
#pragma unroll
    for (int i = 0; i < 6; i++) a[i] = (lane < 6) ? Hs[i * 6 + lane] : 0.0;
    double dmax = (lane < 6) ? sel6(a, lj) : 0.0;
    dmax = fmax(dmax, shfl_xor(dmax, 1));
    dmax = fmax(dmax, shfl_xor(dmax, 2));
    dmax = fmax(dmax, shfl_xor(dmax, 4));
    dmax = shfl(dmax, 0);
    const double thr = dmax * 1e-12;
    bool ok = (dmax > 0.0) && (dmax == dmax) && (dmax < 1e300);
    double rinv[6], dprod = 1.0, dlog = 0.0;   // product of the pivots, rescaled through dlog when it leaves [1e-100, 1e100]
#pragma unroll
    for (int k = 0; k < 6; k++) {
        const double d = shfl(a[k], k);
        ok = ok && (d > thr);
        if (lad) {
            dprod *= fmax(d, 1e-300);
            if (dprod > 1e100 || dprod < 1e-100) { dlog += log(dprod); dprod = 1.0; }
        }
        const double r = rsqrt(fmax(d, 1e-300));
        rinv[k] = r;
        double lk[6];
#pragma unroll
        for (int i = 0; i < 6; i++) lk[i] = (i >= k) ? shfl(a[i], k) * r : 0.0;    // column k of L, everywhere
        const double ljk = sel6(lk, lj);                                            // L[lane][k]
        if (lane > k && lane < 6) {
#pragma unroll
            for (int i = k + 1; i < 6; i++) a[i] -= lk[i] * ljk;
        }
        if (lane == k) {
#pragma unroll
            for (int i = 0; i < 6; i++) a[i] = lk[i];
        }
    }
    double y[6];
#pragma unroll
    for (int k = 0; k < 6; k++) {          // L y = g
        double s = gs[k];
#pragma unroll
        for (int j = 0; j < k; j++) s -= shfl(a[k], j) * y[j];
        y[k] = s * rinv[k];
    }
#pragma unroll
    for (int k = 5; k >= 0; k--) {         // L^T x = y
        double s = y[k];
#pragma unroll
        for (int j = k + 1; j < 6; j++) s -= shfl(a[j], k) * x[j];
        x[k] = s * rinv[k];
    }
    if (lad) *lad = dlog + log(dprod);
    return ok;
}

// Matrix6d::inverse() (partial-pivot LU), src/stereoFrameHandler.cpp:429, :470.  Lanes 0..5 hold the columns of A,
// lanes 6..11 the columns of the identity; row operations are the same in every lane.  Result -> out (shared).
__device__ void warp_inv6(const double* As /* shared row-major */, double* out /* shared row-major */) {
    const int lane = threadIdx.x & 31;
    double a[6];
#pragma unroll
    for (int i = 0; i < 6; i++) a[i] = (lane < 6) ? As[i * 6 + lane] : ((lane - 6 == i) ? 1.0 : 0.0);
#pragma unroll
    for (int k = 0; k < 6; k++) {
        int p = k;
        double big = fabs(a[k]);
#pragma unroll
        for (int i = k + 1; i < 6; i++)
            if (fabs(a[i]) > big) { big = fabs(a[i]); p = i; }
        p = __shfl_sync(FULL_MASK, p, k);          // the pivot row is decided by column k
#pragma unroll
        for (int i = k + 1; i < 6; i++)
            if (p == i) { const double t = a[k]; a[k] = a[i]; a[i] = t; }
        const double piv = shfl(a[k], k);
#pragma unroll
        for (int i = k + 1; i < 6; i++) {
            const double f = shfl(a[i], k) / piv;
            a[i] = (lane == k) ? 0.0 : a[i] - f * a[k];
        }
    }
    double xv[6];
#pragma unroll
    for (int i = 5; i >= 0; i--) {
        double s = a[i];
#pragma unroll
        for (int m = i + 1; m < 6; m++) s -= shfl(a[i], m) * xv[m];
        xv[i] = s / shfl(a[i], i);
    }
    __syncwarp();
    if (lane >= 6 && lane < 12) {
#pragma unroll
        for (int i = 0; i < 6; i++) out[i * 6 + (lane - 6)] = xv[i];
    }
    __syncwarp();
}

// SelfAdjointEigenSolver<Matrix6d>::eigenvalues(): lower triangle, ascending.  Parallel-order Jacobi: the 15 plane
// rotations of a sweep are done as 5 rounds of 3 disjoint rotations (round-robin pairing); lane j holds column j.
__device__ void warp_eig6_sym(const double* Ms /* shared row-major */, double* w /* all lanes: ascending */) {
    const int lane = threadIdx.x & 31;
    const int lj = (lane < 6) ? lane : 0;
    double a[6];
#pragma unroll
    for (int i = 0; i < 6; i++) a[i] = (lane < 6) ? ((i >= lj) ? Ms[i * 6 + lj] : Ms[lj * 6 + i]) : 0.0;
    for (int sweep = 0; sweep < 60; sweep++) {
        double off = 0.0, dg = 0.0;
#pragma unroll
        for (int i = 0; i < 6; i++) {
            const double v = a[i] * a[i];
            if (i == lj) dg += v; else off += v;
        }
        if (lane >= 6) { off = 0.0; dg = 0.0; }
        off = shfl(sum8(off), 0);
        dg = shfl(sum8(dg), 0);
        if (!(off > 1e-22 * dg) || off == 0.0) break;   // quadratic convergence: the eigenvalues are settled to ~1e-16
#pragma unroll
        for (int r = 0; r < 5; r++) {
            // round-robin pairing of {0..5}: partner of lane j in round r (nibble 5-j), and the pairs (p < q)
            int partner, p0, q0, p1, q1, p2, q2;
            if (r == 0) { p0 = 0; q0 = 5; p1 = 1; q1 = 4; p2 = 2; q2 = 3; }
            else if (r == 1) { p0 = 0; q0 = 4; p1 = 3; q1 = 5; p2 = 1; q2 = 2; }
            else if (r == 2) { p0 = 0; q0 = 3; p1 = 2; q1 = 4; p2 = 1; q2 = 5; }
            else if (r == 3) { p0 = 0; q0 = 2; p1 = 1; q1 = 3; p2 = 4; q2 = 5; }
            else { p0 = 0; q0 = 1; p1 = 2; q1 = 5; p2 = 3; q2 = 4; }
            partner = lane;
            if (lane == p0) partner = q0;
            if (lane == q0) partner = p0;
            if (lane == p1) partner = q1;
            if (lane == q1) partner = p1;
            if (lane == p2) partner = q2;
            if (lane == q2) partner = p2;
            const double own_d = sel6(a, lj), other_d = shfl(own_d, partner);
            // A[p][q] as seen by lane p and by lane q drift apart at rounding level; both lanes must derive the
            // SAME angle or the update stops being a rotation: use the symmetrised entry
            const double apq_own = sel6(a, (lane < 6) ? partner : 0);
            const double apq = 0.5 * (apq_own + shfl(apq_own, partner));
            const bool is_p = lane < partner;
            const double app = is_p ? own_d : other_d, aqq = is_p ? other_d : own_d;
            double cs = 1.0, sn = 0.0;
            if (lane < 6 && apq != 0.0) {
                const double tau = (aqq - app) / (2.0 * apq);
                const double t = (tau >= 0.0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1.0 + tau * tau));
                cs = 1.0 / sqrt(1.0 + t * t);
                sn = t * cs;
            }
#pragma unroll
            for (int i = 0; i < 6; i++) {   // columns p, q  (A <- A J)
                const double o = shfl(a[i], partner);
                a[i] = is_p ? (cs * a[i] - sn * o) : (sn * o + cs * a[i]);
            }
            {   // rows p, q of every column  (A <- J^T A), the three disjoint planes of this round
                const double c0 = shfl(cs, p0), s0 = shfl(sn, p0), c1 = shfl(cs, p1), s1 = shfl(sn, p1),
                             c2 = shfl(cs, p2), s2 = shfl(sn, p2);
                double ap = a[p0], aq = a[q0];
                a[p0] = c0 * ap - s0 * aq; a[q0] = s0 * ap + c0 * aq;
                ap = a[p1]; aq = a[q1];
                a[p1] = c1 * ap - s1 * aq; a[q1] = s1 * ap + c1 * aq;
                ap = a[p2]; aq = a[q2];
                a[p2] = c2 * ap - s2 * aq; a[q2] = s2 * ap + c2 * aq;
            }
        }
    }
    const double dj = sel6(a, lj);
#pragma unroll
    for (int i = 0; i < 6; i++) w[i] = shfl(dj, i);
#pragma unroll
    for (int i = 1; i < 6; i++)   // insertion sort, static network; NaNs are left where they are
#pragma unroll
        for (int j = i; j > 0; j--) {
            const double lo = fmin(w[j - 1], w[j]), hi = fmax(w[j - 1], w[j]);
            const bool nanv = (w[j - 1] != w[j - 1]) || (w[j] != w[j]);
            if (!nanv) { w[j - 1] = lo; w[j] = hi; }
        }
}

// isGoodSolution (src/stereoFrameHandler.cpp:292-305); one warp, every lane returns the verdict
// The verdict on the covariance without the eigenvalue iteration, when it is beyond doubt: a symmetric matrix (lower triangle,
// like the eigen solver reads it) whose Cholesky pivots are all safely positive has lambda_min > 0, and a positive definite
// matrix has lambda_max < trace.  So pivots > 1e-10 max(diag) and trace < 1 put every eigenvalue inside (0, 1): the test of
// :296-297 passes whatever the iteration's rounding.  Anything else (indefinite, near-singular, large, NaN) is left to the
// full decomposition.  Every lane runs the same ~60 flops on registers.
__device__ __forceinline__ bool cov_surely_inside_unit(const double* A) {
    double tr = 0.0, dmax = 0.0;
#pragma unroll
    for (int i = 0; i < 6; i++) {
        tr += A[i * 6 + i];
        dmax = fmax(dmax, A[i * 6 + i]);
    }
    if (!(tr < 1.0) || !(dmax > 0.0)) return false;
    const double thr = 1e-10 * dmax;
    double L[6][6];
    bool ok = true;
#pragma unroll
    for (int j = 0; j < 6; j++) {
        double d = A[j * 6 + j];
#pragma unroll
        for (int k = 0; k < j; k++) d -= L[j][k] * L[j][k];
        ok = ok && (d > thr);
        const double inv = rsqrt(fmax(d, 1e-300));
        L[j][j] = d * inv;
#pragma unroll
        for (int i = j + 1; i < 6; i++) {
            double v = A[i * 6 + j];
#pragma unroll
            for (int k = 0; k < j; k++) v -= L[i][k] * L[j][k];
            L[i][j] = v * inv;
        }
    }
    return ok;
}

__device__ bool warp_is_good_solution(const double* DTs, const double* covs, double err, double* eig_out) {
    double w[6];
    if (!eig_out && cov_surely_inside_unit(covs)) {   // eigenvalues not asked for and the matrix is plainly fine
        w[0] = 0.0;
        w[5] = 0.0;
    } else {
        warp_eig6_sym(covs, w);
    }
    if (eig_out) {
#pragma unroll
        for (int i = 0; i < 6; i++) eig_out[i] = w[i];
    }
    bool finite = true;
#pragma unroll
    for (int i = 0; i < 16; i++) {
        const double d = DTs[i] - DTs[i];
        finite = finite && (d == d);
    }
    return !(w[0] < 0.0 || w[5] > 1.0 || err < 0.0 || err > 1.0 || !finite);
}

// ---- per-feature arithmetic --------------------------------------------------------------------------
struct Cam {
    double fx, fy, cx, cy;
};

__device__ __forceinline__ void transform(const double* DT, double x, double y, double z, double& X, double& Y, double& Z) {
    X = (DT[0] * x + DT[1] * y + DT[2] * z) + DT[3];   // DT.block(0,0,3,3) * P + DT.col(3).head(3)  (:567)
    Y = (DT[4] * x + DT[5] * y + DT[6] * z) + DT[7];
    Z = (DT[8] * x + DT[9] * y + DT[10] * z) + DT[11];
}

// residual norm of point i; also the quantities the Jacobian needs
__device__ __forceinline__ double point_residual(const Feat& f, int i, const double* DT, const Cam& c, double& X,
                                                 double& Y, double& Z, double& iz, double& dx, double& dy) {
    transform(DT, f.Px[i], f.Py[i], f.Pz[i], X, Y, Z);
    iz = 1.0 / Z;
    dx = (c.cx + (c.fx * X) * iz) - f.pu[i];   // PinholeStereoCamera::projection (src/pinholeStereoCamera.cpp:231-237)
    dy = (c.cy + (c.fy * Y) * iz) - f.pv[i];
    return sqrt(dx * dx + dy * dy);
}

struct LineRes {
    double sX, sY, sZ, eX, eY, eZ, isz, iez, spu, spv, epu, epv, ds, de;
};

__device__ __forceinline__ double line_residual(const Feat& f, int i, const double* DT, const Cam& c, LineRes& r) {
    transform(DT, f.sX[i], f.sY[i], f.sZ[i], r.sX, r.sY, r.sZ);
    transform(DT, f.eX[i], f.eY[i], f.eZ[i], r.eX, r.eY, r.eZ);
    r.isz = 1.0 / r.sZ;
    r.iez = 1.0 / r.eZ;
    r.spu = c.cx + (c.fx * r.sX) * r.isz;
    r.spv = c.cy + (c.fy * r.sY) * r.isz;
    r.epu = c.cx + (c.fx * r.eX) * r.iez;
    r.epv = c.cy + (c.fy * r.eY) * r.iez;
    const double l0 = f.l0[i], l1 = f.l1[i], l2 = f.l2[i];
    r.ds = l0 * r.spu + l1 * r.spv + l2;   // :621-622
    r.de = l0 * r.epu + l1 * r.epv + l2;
    return sqrt(r.ds * r.ds + r.de * r.de);
}

// fx / max(homogTh, Z^2) (:577) with the reciprocal of Z already at hand
__device__ __forceinline__ double fgz2_of(double fx, double Z, double iz, double th) {
    const double zz = Z * Z;
    return (zz > th) ? (fx * iz) * iz : fx / th;
}

// the 6-vector of :582-587 / :636-641 scaled by `sc` (fgz2 and 1/max(homogTh,|e|) folded in by the caller)
__device__ __forceinline__ void jac_aux(double sc, double gx, double gy, double gz, double dx, double dy, double* J) {
    J[0] = +sc * dx * gz;
    J[1] = +sc * dy * gz;
    J[2] = -sc * (gx * dx + gy * dy);
    J[3] = -sc * (gx * gy * dx + gy * gy * dy + gz * gz * dy);
    J[4] = +sc * (gx * gx * dx + gz * gz * dx + gx * gy * dy);
    J[5] = +sc * (gx * gz * dy - gy * gz * dx);
}

__device__ __forceinline__ double overlap_from_lambdas(double ls, double le) {
    const double lo = (le < ls) ? le : ls, hi = (ls < le) ? le : ls;
    if (lo < 0.0 && hi > 1.0) return 1.0;
    if (hi < 0.0 || lo > 1.0) return 0.0;
    if (lo < 0.0) return hi;
    if (hi > 1.0) return 1.0 - lo;
    return hi - lo;
}

// StereoFrame::lineSegmentOverlap (src/stereoFrame.cpp:510-616): for a fixed previous-frame segment (spl, epl) the
// parameter lambda of a projected endpoint (u, v) is affine in (u, v) in all three branches; the coefficients are
// computed once per matched line when the list is built.
__device__ __forceinline__ void overlap_coeffs(double su, double sv, double eu, double ev, double& oa, double& ob,
                                               double& oc) {
    const double lx = eu - su, ly = ev - sv;
    if (fabs(su - eu) < 1.0) {          // vertical (:515-544): lambda = (v - sv) / ly
        oa = 0.0; ob = 1.0 / ly; oc = -sv / ly;
    } else if (fabs(sv - ev) < 1.0) {   // horizontal (:545-574): lambda = (u - su) / lx
        oa = 1.0 / lx; ob = 0.0; oc = -su / lx;
    } else {                            // generic (:575-612): foot of the perpendicular, then (x - su) / lx
        const double a = sv - ev, b = eu - su, c = su * ev - eu * sv;
        const double lxy = 1.0 / (a * a + b * b);
        oa = (b * b * lxy) / lx;
        ob = (-(a * b) * lxy) / lx;
        oc = (-(a * c) * lxy - su) / lx;
    }
}

__device__ __forceinline__ void accumulate(double* acc, const double* J, double r, double w) {
    int k = 0;
#pragma unroll
    for (int i = 0; i < 6; i++) {
        const double Jw = J[i] * w;
#pragma unroll
        for (int j = i; j < 6; j++) acc[k++] += Jw * J[j];
        acc[21 + i] += Jw * r;
    }
    acc[27] += r * r * w;
    acc[28] += 1.0;
}

// Transposed warp reduction: 32 values per lane -> lane L ends with the warp total of element L (31 shuffles
// instead of 5 per element).  Fixed order: deterministic.
__device__ __forceinline__ double warp_reduce_32(double* v, int lane) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        const bool up = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < off; i++) {
            const double mine = up ? v[i + off] : v[i];
            const double send = up ? v[i] : v[i + off];
            v[i] = mine + shfl_xor(send, off);
        }
    }
    return v[0];
}

// block-wide sums of the per-thread accumulators -> st.acc[0..28]
__device__ void block_reduce_acc(State& st, double* acc) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double mine = warp_reduce_32(acc, lane);
    st.red[warp][lane] = mine;
    __syncthreads();
    if (tid < 32) {
        double s = 0.0;
        const int nw = blockDim.x >> 5;
#pragma unroll
        for (int w = 0; w < K2_WARPS; w++) s += (w < nw) ? st.red[w][tid] : 0.0;
        st.acc[tid] = s;
    }
    __syncthreads();
}

// up to 4 block-wide sums at once (fixed order)
template <int N>
__device__ void block_sum(State& st, double* v) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int k = 0; k < N; k++)
#pragma unroll
        for (int o = 16; o; o >>= 1) v[k] += shfl_xor(v[k], o);
    __syncthreads();
    if (lane == 0)
#pragma unroll
        for (int k = 0; k < N; k++) st.sum[warp][k] = v[k];
    __syncthreads();
    const int nw = blockDim.x >> 5;
#pragma unroll
    for (int k = 0; k < N; k++) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < K2_WARPS; w++) s += (w < nw) ? st.sum[w][k] : 0.0;
        v[k] = s;
    }
}

// ---- bitonic sort of a[0..m) in shared memory, m a power of two >= 32 ------------------------------------------
// Fast path (128 <= m <= 4 * blockDim): thread t keeps positions 4t..4t+3 in registers; strides 1, 2 are in-thread,
// strides 4..64 are warp shuffles, only strides >= 128 go through shared memory with a block barrier.
__device__ void bitonic_sort_smem(double* a, int m) {   // generic path: every stride through shared memory
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int seg = max(m / K2_WARPS, 32);
    const int nseg = m / seg;
    const int base = warp * seg;
    __syncthreads();
    for (int k = 2; k <= m; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (warp < nseg) {
                for (int e = lane; e < seg; e += 32) {
                    const int i = base + e, ixj = i ^ j;
                    if (ixj > i) {
                        const double x = a[i], y = a[ixj];
                        const bool up = ((i & k) == 0);
                        if ((x > y) == up) {
                            a[i] = y;
                            a[ixj] = x;
                        }
                    }
                }
            }
            const int next = (j > 1) ? (j >> 1) : k;   // stride of the following stage
            if (j >= seg || next >= seg) __syncthreads();
            else __syncwarp();
        }
    }
    __syncthreads();
}

__device__ __forceinline__ void cmpx(double& x, double& y, bool up) {   // (x, y) -> ascending if up
    const double lo = fmin(x, y), hi = fmax(x, y);
    x = up ? lo : hi;
    y = up ? hi : lo;
}

__device__ void bitonic_sort(double* a, int m) {
    const int tid = threadIdx.x, nth = blockDim.x;
    if (m < 128 || m > 4 * nth) {
        bitonic_sort_smem(a, m);
        return;
    }
    const bool active = tid < (m >> 2);      // whole warps: m / 4 is a multiple of 32
    __syncthreads();
    double v[4];
    if (active) {
        const double2 p0 = *reinterpret_cast<const double2*>(a + 4 * tid);
        const double2 p1 = *reinterpret_cast<const double2*>(a + 4 * tid + 2);
        v[0] = p0.x; v[1] = p0.y; v[2] = p1.x; v[3] = p1.y;
    }
    for (int k = 2; k <= m; k <<= 1) {
        int j = k >> 1;
        if (j >= 128) {                       // strides that cross warps: through shared memory
            if (active) {
                *reinterpret_cast<double2*>(a + 4 * tid) = make_double2(v[0], v[1]);
                *reinterpret_cast<double2*>(a + 4 * tid + 2) = make_double2(v[2], v[3]);
            }
            __syncthreads();
            for (; j >= 128; j >>= 1) {
                for (int p = tid; p < (m >> 1); p += nth) {
                    const int i = ((p & ~(j - 1)) << 1) | (p & (j - 1)), ixj = i | j;
                    const double x = a[i], y = a[ixj];
                    const bool up = ((i & k) == 0);
                    if ((x > y) == up) {
                        a[i] = y;
                        a[ixj] = x;
                    }
                }
                __syncthreads();
            }
            if (active) {
                const double2 p0 = *reinterpret_cast<const double2*>(a + 4 * tid);
                const double2 p1 = *reinterpret_cast<const double2*>(a + 4 * tid + 2);
                v[0] = p0.x; v[1] = p0.y; v[2] = p1.x; v[3] = p1.y;
            }
        }
        if (active) {
            const int i0 = 4 * tid;
            for (; j >= 4; j >>= 1) {         // partner in another lane of this warp
                const int lm = j >> 2;
                const bool up = ((i0 & k) == 0), lower = ((i0 & j) == 0);   // bits >= 2: the same for all four
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    const double y = shfl_xor(v[e], lm);
                    v[e] = (lower == up) ? fmin(v[e], y) : fmax(v[e], y);
                }
            }
            if (k >= 4) {                     // stride 2: (0,2) (1,3)
                const bool up = ((i0 & k) == 0);
                cmpx(v[0], v[2], up);
                cmpx(v[1], v[3], up);
            }
            {                                 // stride 1: (0,1) (2,3)
                const bool up0 = (((i0) & k) == 0), up2 = (((i0 + 2) & k) == 0);
                cmpx(v[0], v[1], up0);
                cmpx(v[2], v[3], up2);
            }
        }
    }
    if (active) {
        *reinterpret_cast<double2*>(a + 4 * tid) = make_double2(v[0], v[1]);
        *reinterpret_cast<double2*>(a + 4 * tid + 2) = make_double2(v[2], v[3]);
    }
    __syncthreads();
}

__device__ __forceinline__ int pow2_ceil(int n) {
    int m = 1;
    while (m < n) m <<= 1;
    return m;
}

// ---- keys whose unsigned order is the numeric order of the doubles they come from ----
__device__ __forceinline__ unsigned long long select_key(double x) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(x);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double select_unkey(unsigned long long k) {
    return __longlong_as_double((long long)((k >> 63) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k));
}
// ---- k-th smallest of val(0 .. m) by radix selection with 11-bit digits, for the streamed solver's lists ------------------------------------
// Keys of one list share their sign / exponent bits, so the digits start below the common prefix of the smallest and the
// largest key; one 2048-bin histogram then usually leaves a handful of candidates around rank k, which are ranked against
// each other directly.  Typical cost: one min / max reduction + one histogram pass + one gather (a byte-wise radix selection
// needs three to four passes and a fetch).  K2 keeps its bitonic sort: at 2000 entries and 512 threads the sort (register /
// shuffle strides) is as fast as four selections, and for the robust solver's per-iteration MAD at 1000 entries it is faster
// (measured: C3 K2 1.87 ms with the sort, 2.04 ms with selections).  Scratch: SEL_BINS ints + SEL_CAND keys + 8 ints of shared memory.
constexpr int SEL_BITS = 11, SEL_BINS = 1 << SEL_BITS, SEL_CAND = 256;
struct SelScratch {
    int* hist;                     // [SEL_BINS]
    unsigned long long* cand;      // [SEL_CAND]
    int* ctl;                      // [8]
};
__host__ __device__ inline size_t sel_scratch_bytes() { return (size_t)SEL_BINS * 4 + (size_t)SEL_CAND * 8 + 64; }
__device__ __forceinline__ SelScratch sel_scratch_at(uint8_t* base) {   // base 16-byte aligned
    SelScratch sc;
    sc.cand = reinterpret_cast<unsigned long long*>(base);
    sc.hist = reinterpret_cast<int*>(base + (size_t)SEL_CAND * 8);
    sc.ctl = sc.hist + SEL_BINS;
    return sc;
}
template <class Val>
__device__ double block_select_wide(const SelScratch& sc, State& st, int m, int k, Val val) {
    const int tid = threadIdx.x, nth = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nth >> 5;
    unsigned long long lo = ~0ull, hi = 0ull;
    for (int i = tid; i < m; i += nth) {
        const unsigned long long key = select_key(val(i));
        lo = key < lo ? key : lo;
        hi = key > hi ? key : hi;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const unsigned long long l2 = __shfl_xor_sync(FULL_MASK, lo, o), h2 = __shfl_xor_sync(FULL_MASK, hi, o);
        lo = l2 < lo ? l2 : lo;
        hi = h2 > hi ? h2 : hi;
    }
    unsigned long long* mm = reinterpret_cast<unsigned long long*>(&st.red[0][0]);
    __syncthreads();
    if (lane == 0) { mm[2 * warp] = lo; mm[2 * warp + 1] = hi; }
    __syncthreads();
    for (int w = 0; w < nw; w++) {
        const unsigned long long l2 = mm[2 * w], h2 = mm[2 * w + 1];
        lo = l2 < lo ? l2 : lo;
        hi = h2 > hi ? h2 : hi;
    }
    __syncthreads();
    if (lo == hi) return select_unkey(lo);
    int hb = 64 - __clzll((long long)(lo ^ hi));      // undecided low bits: everything above is common to all keys
    unsigned long long prefix = (hb >= 64) ? 0ull : ((hi >> hb) << hb);
    int kk = k;
    double result = 0.0;
    for (;;) {
        const int bits = hb < SEL_BITS ? hb : SEL_BITS, sh = hb - bits, nb = 1 << bits;
        for (int b = tid; b < nb; b += nth) sc.hist[b] = 0;
        __syncthreads();
        for (int i = tid; i < m; i += nth) {
            const unsigned long long key = select_key(val(i));
            const bool under = (hb >= 64) || ((key >> hb) == (prefix >> hb));
            if (under) atomicAdd(&sc.hist[(unsigned)(key >> sh) & (unsigned)(nb - 1)], 1);
        }
        __syncthreads();
        {   // the bin that holds rank kk: a run of bins per thread, block scan over the run sums, a short walk inside the run
            const int per = (nb + nth - 1) / nth, b0 = tid * per;
            int sum = 0;
            for (int j = 0; j < per; j++) sum += (b0 + j < nb) ? sc.hist[b0 + j] : 0;
            int inc = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(FULL_MASK, inc, o);
                if (lane >= o) inc += t;
            }
            if (lane == 31) st.scan[warp] = inc;
            __syncthreads();
            int base = 0;
            for (int w = 0; w < warp; w++) base += st.scan[w];
            const int excl = base + inc - sum;
            if (kk >= excl && kk < excl + sum) {
                int before = excl, j = 0;
                while (before + sc.hist[b0 + j] <= kk) { before += sc.hist[b0 + j]; j++; }
                sc.ctl[0] = b0 + j;
                sc.ctl[1] = kk - before;
                sc.ctl[2] = sc.hist[b0 + j];
                sc.ctl[3] = 0;
            }
            __syncthreads();
        }
        const int bin = sc.ctl[0], cnt = sc.ctl[2];
        kk = sc.ctl[1];
        prefix |= (unsigned long long)(unsigned)bin << sh;
        hb = sh;
        if (hb == 0) {                    // every bit decided: the cnt keys left are all equal to the prefix
            result = select_unkey(prefix);
            break;
        }
        if (cnt <= SEL_CAND) {            // few keys left under the prefix: rank them against each other
            for (int i = tid; i < m; i += nth) {
                const unsigned long long key = select_key(val(i));
                if ((key >> hb) == (prefix >> hb)) sc.cand[atomicAdd(&sc.ctl[3], 1)] = key;
            }
            __syncthreads();
            for (int c = tid; c < cnt; c += nth) {
                const unsigned long long mine = sc.cand[c];
                int less = 0, eq = 0;
                for (int j = 0; j < cnt; j++) {
                    const unsigned long long o = sc.cand[j];
                    less += (o < mine) ? 1 : 0;
                    eq += (o == mine) ? 1 : 0;
                }
                if (kk >= less && kk < less + eq) {   // equal keys all write the same value
                    sc.ctl[4] = (int)(unsigned)(mine & 0xFFFFFFFFull);
                    sc.ctl[5] = (int)(unsigned)(mine >> 32);
                }
            }
            __syncthreads();
            result = select_unkey(((unsigned long long)(unsigned)sc.ctl[5] << 32) | (unsigned long long)(unsigned)sc.ctl[4]);
            break;
        }
        __syncthreads();                  // ctl / hist are rewritten by the next digit
    }
    __syncthreads();
    return result;
}

// median / MAD of the n finite values in `buf` SORTED ascending (+inf padding behind them):
// median = sorted[n/2]; stdv = 1.4826 * sorted(|x - median| rounded to float)[n/2]  (src/auxiliar.cpp:396-403).
// The deviations of a sorted array form a V (non-increasing up to the median, non-decreasing after it): their n/2-th
// smallest is the k-th element of the union of two sorted runs, found by binary search by every thread on its own.
__device__ void median_mad(const double* buf, int n, double& median, double& stdv) {
    const int h = n / 2;
    const double med = buf[h];
    const int nL = h + 1, nR = n - h - 1, k = h;      // left run: buf[h], buf[h-1], ...; right run: buf[h+1], ...
    auto dev = [&](int idx) -> double { return (double)fabsf((float)(buf[idx] - med)); };
    auto Lat = [&](int i) -> double { return (i < 0) ? -INFINITY : (i >= nL ? INFINITY : dev(h - i)); };
    auto Rat = [&](int i) -> double { return (i < 0) ? -INFINITY : (i >= nR ? INFINITY : dev(h + 1 + i)); };
    // a = how many of the k+1 smallest deviations come from the left run: smallest a with L[a] >= R[k - a]
    int lo = max(0, k + 1 - nR), hi = min(k + 1, nL);
    while (lo < hi) {
        const int a = (lo + hi) >> 1;
        if (Lat(a) < Rat(k - a)) lo = a + 1;
        else hi = a;
    }
    const double mad = fmax(Lat(lo - 1), Rat(k - lo));
    median = med;
    stdv = 1.4826 * mad;
}

// ---- optimizeFunctions / optimizeFunctionsRobust -------------------------------------------------------
// pre-weight pass + MAD scales (src/stereoFrameHandler.cpp:707-781)
__device__ void robust_scales(const Feat& f, State& st, double* sortbuf, const double* DT, const Cam& cam,
                              double& s_p, double& s_l) {
    const int tid = threadIdx.x, nth = blockDim.x;
    const double th_min = 0.0001, th_max = sqrt(7.815);
    double sc[2];
    for (int type = 0; type < 2; type++) {
        const int nn = type ? f.nl : f.np;
        const int m = pow2_ceil(max(nn, 32));
        double cnt[1] = {0.0};
        for (int i = tid; i < m; i += nth) {
            double v = INFINITY;
            if (i < nn && (type ? f.inl_l[i] : f.inl_p[i])) {
                if (type == 0) {
                    double X, Y, Z, iz, dx, dy;
                    v = point_residual(f, i, DT, cam, X, Y, Z, iz, dx, dy);
                } else {
                    LineRes r;
                    v = line_residual(f, i, DT, cam, r);
                }
                cnt[0] += 1.0;
            }
            sortbuf[i] = v;
        }
        block_sum<1>(st, cnt);                       // res.size(): the inliers only (:710-739)
        const int n = (int)cnt[0];
        double s = 0.0;                              // vector_stdv_mad of an empty vector
        if (n > 0) {
            bitonic_sort(sortbuf, m);
            double med;
            median_mad(sortbuf, n, med, s);
        }
        __syncthreads();
        sc[type] = fmin(fmax(s, th_min), th_max);
    }
    s_p = sc[0];
    s_l = sc[1];
}

// leaves the reduced sums in st.acc (H upper triangle, g, e, N)
__device__ void evaluate(const Feat& f, State& st, double* sortbuf, const double* DT, const Cam& cam,
                         double homog_th, bool robust) {
    const int tid = threadIdx.x, nth = blockDim.x;
    double is_p = 1.0, is_l = 1.0;
    if (robust) {
        double s_p, s_l;
        robust_scales(f, st, sortbuf, DT, cam, s_p, s_l);
        is_p = 1.0 / s_p;
        is_l = 1.0 / s_l;
    }
    double acc[32];
#pragma unroll
    for (int k = 0; k < 32; k++) acc[k] = 0.0;

    for (int i = tid; i < f.np; i += nth) {   // point block (:563-606 / :785-870)
        if (!f.inl_p[i]) continue;
        double X, Y, Z, iz, dx, dy, J[6];
        const double n = point_residual(f, i, DT, cam, X, Y, Z, iz, dx, dy);
        const double sc = fgz2_of(cam.fx, Z, iz, homog_th) / fmax(homog_th, n);   // fgz2 / max(homogTh, |e|)
        jac_aux(sc, X, Y, Z, dx, dy, J);
        double r, w;
        if (!robust) {
            r = n * f.pss[i];                   // |e| sqrt(sigma2)  (:591)
            w = 1.0 / (1.0 + r * r);            // robustWeightCauchy (src/auxiliar.cpp:556-559)
        } else {
            r = n;
            const double x = r * is_p;
            w = 1.0 / (1.0 + x * x);
        }
        accumulate(acc, J, r, w);
    }
    for (int i = tid; i < f.nl; i += nth) {   // line block (:610-684 / :874-952)
        if (!f.inl_l[i]) continue;
        LineRes lr;
        double Js[6], Je[6], J[6];
        const double n = line_residual(f, i, DT, cam, lr);
        const double lx = f.l0[i], ly = f.l1[i];
        const double iden = 1.0 / fmax(homog_th, n);
        jac_aux(fgz2_of(cam.fx, lr.sZ, lr.isz, homog_th) * lr.ds * iden, lr.sX, lr.sY, lr.sZ, lx, ly, Js);
        jac_aux(fgz2_of(cam.fx, lr.eZ, lr.iez, homog_th) * lr.de * iden, lr.eX, lr.eY, lr.eZ, lx, ly, Je);
#pragma unroll
        for (int k = 0; k < 6; k++) J[k] = Js[k] + Je[k];                          // (Js ds + Je de) / max(homogTh, |e|)
        double r, w;
        if (!robust) {
            r = n * f.lss[i];
            w = 1.0 / (1.0 + r * r);
        } else {
            r = n;
            const double x = r * is_l;
            w = 1.0 / (1.0 + x * x);
        }
        const double oa = f.oa[i], ob = f.ob[i], oc = f.oc[i];                     // overlap with the PREVIOUS segment (:668)
        w *= overlap_from_lambdas(oa * lr.spu + ob * lr.spv + oc, oa * lr.epu + ob * lr.epv + oc);
        accumulate(acc, J, r, w);
    }
    block_reduce_acc(st, acc);
}

// warp 0: st.acc -> st.H (full symmetric); returns err = e / N
__device__ __forceinline__ double unpack_normal_equations(State& st, int lane) {
    if (lane < 6) {
#pragma unroll
        for (int i = 0; i < 6; i++) {
            const int lo = min(i, lane), hi = max(i, lane);
            st.H[i * 6 + lane] = st.acc[tri(lo, hi)];
        }
    }
    __syncwarp();
    return st.acc[27] / st.acc[28];   // e /= (N_l + N_p)  (:692)
}

// warp 0: DT << DT * inverse_se3(expmap_se3(inc))  (:419); every lane computes, lanes 0..15 store
__device__ __forceinline__ void apply_increment(double* DTs, const double* inc, int lane) {
    double E[16], Ei[16], D[16], R[16];
    expmap_se3(inc, E);
    inverse_se3(E, Ei);
#pragma unroll
    for (int i = 0; i < 16; i++) D[i] = DTs[i];
    mat4_mul(D, Ei, R);
    __syncwarp();
    double mine = R[0];
#pragma unroll
    for (int i = 1; i < 16; i++) mine = (lane == i) ? R[i] : mine;
    if (lane < 16) DTs[lane] = mine;
    __syncwarp();
}

// gaussNewtonOptimization (:394-431) and gaussNewtonOptimizationRobust (:433-480).
// Pose in st.DT (in/out), covariance to st.cov, error to st.err.  Block-wide; warp 0 runs the 6x6 part.
__device__ void gauss_newton(const Feat& f, State& st, double* sortbuf, const Cam& cam, const PlConfig& cfg,
                             int max_iters, bool robust) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double err_prev = 999999999.9, err = 0.0;   // warp 0's copies are the authoritative ones (uniform across its lanes)
    bool good = true, fail_first = false;
    double DTstart = 0.0;                       // lane i < 16 of warp 0 keeps entry i of the initial pose
    if (warp == 0) {
        if (lane < 16) DTstart = st.DT[lane];
        for (int i = lane; i < 36; i += 32) st.H[i] = 0.0;
        if (lane == 0) st.evals = 0;
    }
    for (int it = 0; it < max_iters; it++) {
        const long long t_a = clock64();
        evaluate(f, st, sortbuf, st.DT, cam, cfg.homog_th, robust);
        const long long t_b = clock64();
        if (warp == 0) {
            double inc[6], lad;
            int ctrl = 0;   // 0 continue, 1 stop
            err = unpack_normal_equations(st, lane);
            if (!robust) {
                if (err > err_prev) {
                    ctrl = 1;
                    if (it == 0) fail_first = true;
                } else if ((err < cfg.min_error) || fabs(err - err_prev) < cfg.min_error_change) {
                    ctrl = 1;
                } else {
                    if (!warp_chol6_solve(st.H, &st.acc[21], inc)) warp_qr6_solve<false>(st.H, &st.acc[21], inc, lad);
                    apply_increment(st.DT, inc, lane);
                    if (sqrt(inc[0] * inc[0] + inc[1] * inc[1] + inc[2] * inc[2]) < cfg.min_error_change &&
                        sqrt(inc[3] * inc[3] + inc[4] * inc[4] + inc[5] * inc[5]) < cfg.min_error_change)
                        ctrl = 1;
                    err_prev = err;
                }
            } else {
                if ((fabs(err - err_prev) < cfg.min_error_change) || (err < cfg.min_error)) {
                    ctrl = 1;
                } else {
                    // SPD normal equations (the regular case): Cholesky gives the increment and log|det| for a tenth of the
                    // pivoted QR's cycles; anything else goes through the QR like the reference
                    if (!warp_chol6_solve(st.H, &st.acc[21], inc, &lad)) warp_qr6_solve<true>(st.H, &st.acc[21], inc, lad);
                    if (lad < 0.0) {
                        good = false;
                        ctrl = 1;
                    } else {
                        apply_increment(st.DT, inc, lane);
                        double n2 = 0.0;
#pragma unroll
                        for (int i = 0; i < 6; i++) n2 += inc[i] * inc[i];
                        if (sqrt(n2) < cfg.min_error_change) ctrl = 1;
                        err_prev = err;
                    }
                }
            }
            if (lane == 0) {
                st.ctrl = ctrl;
                st.evals++;
                st.tc[2] += t_b - t_a;
                st.tc[3] += clock64() - t_b;
            }
        }
        __syncthreads();
        const int ctrl = st.ctrl;
        __syncthreads();
        if (ctrl) break;
    }
    if (warp == 0) {
        const long long t_c = clock64();
        if (fail_first) {
            if (lane == 0) st.err = -1.0;   // :408-409: DT_cov left untouched
        } else if (good) {
            warp_inv6(st.H, st.cov);
            if (lane == 0) st.err = err;
        } else {   // :473-478
            if (lane < 16) st.DT[lane] = DTstart;
            if (lane == 0) st.err = -1.0;
            for (int i = lane; i < 36; i += 32) st.cov[i] = (i % 7 == 0) ? 1.0 : 0.0;
        }
        if (lane == 0) st.tc[3] += clock64() - t_c;
    }
    __syncthreads();
}

// removeOutliers (:988-1067) for LONG lists (the streamed solver: 8000 + 2000 entries): res_pt(i) / res_ls(i) = |e| sqrt(sigma2)
// of matched feature i at the stage-1 pose, each formed ONCE, straight into shared memory; median and MAD by radix selection
// (a full bitonic sort of 8192 doubles through shared memory costs 10x more).  Same order statistics, same flags as
// remove_outliers.  `points_filled`: the caller has already put the point residuals into sortbuf.  drop_pt(i) / drop_ls(i): told
// of every flag that goes from 1 to 0 (the streamed solver clears the flag inside its fp32 record there).
template <class ResP, class ResL, class DropP, class DropL>
__device__ void remove_outliers_select(const Feat& f, State& st, double* sortbuf, const SelScratch& sel, const PlConfig& cfg,
                                       bool points_filled, ResP res_pt, ResL res_ls, DropP drop_pt, DropL drop_ls) {
    const int tid = threadIdx.x, nth = blockDim.x;
    for (int type = 0; type < 2; type++) {
        const int n = type ? f.nl : f.np;
        if (type == 0 ? !cfg.has_points : !cfg.has_lines) continue;
        if (n == 0) continue;   // vector_mean_stdv_mad of an empty vector: nothing to flag
        // residuals of ALL matched features (inliers or not)
        if (type == 1) {
#pragma unroll 2
            for (int i = tid; i < n; i += nth) sortbuf[i] = res_ls(i);
        } else if (!points_filled) {
#pragma unroll 4
            for (int i = tid; i < n; i += nth) sortbuf[i] = res_pt(i);
        }
        __syncthreads();
        auto residual = [&](int i) -> double { return sortbuf[i]; };
        const long long t_s = clock64();
        // median = sorted[n / 2]; stdv = 1.4826 * sorted(|x - median| rounded to float)[n / 2]  (src/auxiliar.cpp:396-403):
        // two order statistics, no sort
        const double median = block_select_wide(sel, st, n, n / 2, residual);
        const double mad = block_select_wide(sel, st, n, n / 2, [&](int i) -> double { return (double)fabsf((float)(sortbuf[i] - median)); });
        const double stdv = 1.4826 * mad;
        if (tid == 0) st.tc[7] += clock64() - t_s;
        // mean of the residuals below 2 stdv if there are enough of them, else plain mean (auxiliar.cpp:406-427)
        double s[3] = {0.0, 0.0, 0.0};
        for (int i = tid; i < n; i += nth) {
            const double r = residual(i);
            s[2] += r;
            if (r < 2.0 * stdv) {
                s[0] += r;
                s[1] += 1.0;
            }
        }
        block_sum<3>(st, s);
        const int k = (int)s[1];
        const double mean = (k >= (int)(0.2 * (double)n)) ? s[0] / (double)k : s[2] / (double)n;
        const double th = cfg.inlier_k * stdv;
        double removed[1] = {0.0};
        uint8_t* inl = type ? f.inl_l : f.inl_p;
#pragma unroll 4
        for (int i = tid; i < n; i += nth)
            if (fabs(residual(i) - mean) > th && inl[i]) {
                inl[i] = 0;
                removed[0] += 1.0;
                if (type == 0) drop_pt(i); else drop_ls(i);
            }
        block_sum<1>(st, removed);
        if (tid == 0) {
            if (type == 0) st.n_inl_p -= (int)removed[0];
            else st.n_inl_l -= (int)removed[0];
        }
        __syncthreads();
    }
}

// removeOutliers (:988-1067) at pose DT (shared)
__device__ void remove_outliers(const Feat& f, State& st, double* sortbuf, const double* DT, const Cam& cam,
                                const PlConfig& cfg) {
    const int tid = threadIdx.x, nth = blockDim.x;
    for (int type = 0; type < 2; type++) {
        const int n = type ? f.nl : f.np;
        if (type == 0 ? !cfg.has_points : !cfg.has_lines) continue;
        if (n == 0) continue;   // vector_mean_stdv_mad of an empty vector: nothing to flag
        const int m = pow2_ceil(max(n, 32));
        // residuals of ALL matched features (inliers or not), |e| sqrt(sigma2)
        auto residual = [&](int i) -> double {
            if (type == 0) {
                double X, Y, Z, iz, dx, dy;
                return point_residual(f, i, DT, cam, X, Y, Z, iz, dx, dy) * f.pss[i];
            }
            LineRes r;
            return line_residual(f, i, DT, cam, r) * f.lss[i];
        };
        for (int i = tid; i < m; i += nth) sortbuf[i] = (i < n) ? residual(i) : INFINITY;
        const long long t_s = clock64();
        bitonic_sort(sortbuf, m);
        double median, stdv;
        median_mad(sortbuf, n, median, stdv);
        if (tid == 0) st.tc[7] += clock64() - t_s;
        // mean of the residuals below 2 stdv if there are enough of them, else plain mean (auxiliar.cpp:406-427)
        double s[3] = {0.0, 0.0, 0.0};
        for (int i = tid; i < n; i += nth) {
            const double r = residual(i);
            s[2] += r;
            if (r < 2.0 * stdv) {
                s[0] += r;
                s[1] += 1.0;
            }
        }
        block_sum<3>(st, s);
        const int k = (int)s[1];
        const double mean = (k >= (int)(0.2 * (double)n)) ? s[0] / (double)k : s[2] / (double)n;
        const double th = cfg.inlier_k * stdv;
        double removed[1] = {0.0};
        uint8_t* inl = type ? f.inl_l : f.inl_p;
        for (int i = tid; i < n; i += nth)
            if (inl[i] && fabs(residual(i) - mean) > th) {
                inl[i] = 0;
                removed[0] += 1.0;
            }
        block_sum<1>(st, removed);
        if (tid == 0) {
            if (type == 0) st.n_inl_p -= (int)removed[0];
            else st.n_inl_l -= (int)removed[0];
        }
        __syncthreads();
    }
}

// block-wide exclusive scan of one int per thread; returns the thread's offset, total in *total
__device__ int block_exclusive_scan(State& st, int v, int* total) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int inc = v;
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(FULL_MASK, inc, o);
        if (lane >= o) inc += t;
    }
    __syncthreads();
    if (lane == 31) st.scan[warp] = inc;
    __syncthreads();
    int base = 0, tot = 0;
    const int nw = blockDim.x >> 5;
    for (int w = 0; w < nw; w++) {
        if (w < warp) base += st.scan[w];
        tot += st.scan[w];
    }
    *total = tot;
    __syncthreads();
    return base + inc - v;
}

// Pose finalisation (src/stereoFrameHandler.cpp:372-391) by ONE warp: gate, curr->DT = exp(log(inverse(DT))), Tfw chain,
// covariance propagation, eigenvalues; fills st.out.  `phase_out` (optional): the debug phase timers of this pair.
__device__ void finalize_pose(State& st, const PlPrior* prior, const Feat& f, int lane, long long* phase_out) {
        const long long t_f = clock64();
        PlPoseResult& o = st.out;
        double* Tfw_prev = st.red[0];        // 16 doubles of scratch
        double* Tfw_cov_prev = st.red[1];    // 36 doubles (runs into red[2], free here)
        double* Ad = st.red[4];              // 36 doubles (red[4], red[5])
        if (lane < 16) Tfw_prev[lane] = prior ? prior->Tfw[lane] : ((lane % 5 == 0) ? 1.0 : 0.0);
        for (int i = lane; i < 36; i += 32)  // initialize(): Tfw = I, Tfw_cov = I (:43-44)
            Tfw_cov_prev[i] = prior ? prior->Tfw_cov[i] : ((i % 7 == 0) ? 1.0 : 0.0);
        if (lane < 16) o.DT_opt[lane] = st.DT[lane];
        __syncwarp();
        double eig[6], D[16];
#pragma unroll
        for (int i = 0; i < 16; i++) D[i] = st.DT[i];
        const bool ok = warp_is_good_solution(st.DT, st.cov, st.err, eig) && !mat4_is_identity(D);
        if (ok) {
            double Ti[16], x[6], E[16], T2[16], T3[16], P[16];
            inverse_se3(D, Ti);
            logmap_se3(Ti, x);
            expmap_se3(x, E);                                                     // :374
#pragma unroll
            for (int i = 0; i < 16; i++) P[i] = Tfw_prev[i];
            mat4_mul(P, E, T2);
            logmap_se3(T2, x);
            expmap_se3(x, T3);                                                    // :377
            double e_mine = E[0], t_mine = T3[0];
#pragma unroll
            for (int i = 1; i < 16; i++) {
                e_mine = (lane == i) ? E[i] : e_mine;
                t_mine = (lane == i) ? T3[i] : t_mine;
            }
            if (lane < 16) { o.DT[lane] = e_mine; o.Tfw[lane] = t_mine; }
            for (int i = lane; i < 36; i += 32) o.DT_cov[i] = st.cov[i];
            // unccomp_se3 (src/auxiliar.cpp:175-197): cov1 + Ad(T1) covinc Ad(T1)^T, Ad = [R, skew(t) R; 0, R]
            {
                double S[9], R3[9], SR[9];
#pragma unroll
                for (int i = 0; i < 3; i++)
#pragma unroll
                    for (int j = 0; j < 3; j++) R3[i * 3 + j] = P[i * 4 + j];
                skew3(P[3], P[7], P[11], S);
                mat3_mul(S, R3, SR);
                for (int e = lane; e < 36; e += 32) {
                    const int i = e / 6, j = e % 6;
                    double v = 0.0;
                    if (i < 3 && j < 3) v = sel9(R3, i * 3 + j);
                    else if (i < 3 && j >= 3) v = sel9(SR, i * 3 + (j - 3));
                    else if (i >= 3 && j >= 3) v = sel9(R3, (i - 3) * 3 + (j - 3));
                    Ad[e] = v;
                }
            }
            __syncwarp();
            for (int e = lane; e < 36; e += 32) {
                const int i = e / 6, j = e % 6;
                double s = 0.0;
                for (int k = 0; k < 6; k++) {
                    double tk = 0.0;
                    for (int l = 0; l < 6; l++) tk += Ad[i * 6 + l] * st.cov[l * 6 + k];
                    s += tk * Ad[j * 6 + k];
                }
                o.Tfw_cov[e] = Tfw_cov_prev[e] + s;                               // :378
            }
            if (lane < 6) o.DT_cov_eig[lane] = sel6(eig, lane);                   // :379-380
            if (lane == 0) { o.err_norm = st.err; o.good = 1; }
        } else {
            if (lane < 16) { o.DT[lane] = (lane % 5 == 0) ? 1.0 : 0.0; o.Tfw[lane] = Tfw_prev[lane]; }
            for (int i = lane; i < 36; i += 32) { o.DT_cov[i] = 0.0; o.Tfw_cov[i] = Tfw_cov_prev[i]; }
            if (lane < 6) o.DT_cov_eig[lane] = 0.0;
            if (lane == 0) { o.err_norm = -1.0; o.good = 0; }
        }
        if (lane == 0) {
            o.n_matched_pt = f.np;
            o.n_matched_ls = f.nl;
            o.n_inliers_pt = st.n_inl_p;
            o.n_inliers_ls = st.n_inl_l;
            o.n_inliers = st.n_inl_p + st.n_inl_l;
            o.reserved = 0;
            st.tc[6] += clock64() - t_f;
            if (phase_out)
                for (int i = 0; i < 8; i++) phase_out[i] = st.tc[i];
        }
}

// Phases A and B of the per-pair work: finish the matching (ratio test and mutual filter on K1's partials -> m12) and build
// matched_pt / matched_ls in ascending prev index as SoA (f), or copy the caller's explicit lists (mode 1).  Block-wide.
// where the streamed solver wants the fp32 records of the lists (gn_stream.cuh "records"); on = false: fp64 lists only (K2)
struct RecordSink {
    bool on;
    float4* pt;      // first record slot of this problem (tile-planar: [cnt] float4 per plane, GS_PT_TILE / GS_LS_TILE per tile)
    float4* ls;
    GsCamD cam;
};
__device__ __forceinline__ void sink_point(const RecordSink& rs, int k, int np, double x, double y, double z, double u, double v,
                                           double pss, bool inl) {
    const int t = k / GS_PT_TILE, r = k % GS_PT_TILE, cnt = min(GS_PT_TILE, np - t * GS_PT_TILE);
    float4* base = rs.pt + 2 * (size_t)t * GS_PT_TILE;
    gs_pack_point(rs.cam, x, y, z, u, v, pss, inl, base[r], base[cnt + r]);
}
__device__ __forceinline__ void sink_line(const RecordSink& rs, int k, int nl, double sx, double sy, double sz, double ex, double ey,
                                          double ez, double l0, double l1, double l2, double oa, double ob, double oc, double lss,
                                          bool inl) {
    const int t = k / GS_LS_TILE, r = k % GS_LS_TILE, cnt = min(GS_LS_TILE, nl - t * GS_LS_TILE);
    float4* base = rs.ls + 4 * (size_t)t * GS_LS_TILE;
    gs_pack_line(rs.cam, sx, sy, sz, ex, ey, ez, l0, l1, l2, oa, ob, oc, lss, inl, base[r], base[cnt + r], base[2 * cnt + r],
                 base[3 * cnt + r]);
}

// Ordered compaction plan of m12[0 .. n1): cc[ch] = number of matches before 32-feature chunk ch (exclusive prefix), returns the
// total.  One ballot per chunk, ONE block scan in all: the gather loops that follow have no block barrier in them, so their
// dependent global loads (m12 -> the matched curr feature) of different chunks overlap freely.
__device__ int compaction_plan(State& st, const int32_t* __restrict__ m12, int n1, int* cc) {
    const int tid = threadIdx.x, nth = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nth >> 5;
    const int nch = (n1 + 31) >> 5;
    for (int ch = warp; ch < nch; ch += nw) {
        const int i = ch * 32 + lane;
        const unsigned bal = __ballot_sync(FULL_MASK, i < n1 && m12[i] >= 0);
        if (lane == 0) cc[ch] = __popc(bal);
    }
    __syncthreads();
    const int per = (nch + nth - 1) / nth, c0 = tid * per;
    int sum = 0;
    for (int j = 0; j < per; j++) sum += (c0 + j < nch) ? cc[c0 + j] : 0;
    int total;
    int run = block_exclusive_scan(st, sum, &total);      // (barriers inside: every read of cc above is done before the writes below)
    for (int j = 0; j < per; j++)
        if (c0 + j < nch) {
            const int c = cc[c0 + j];
            cc[c0 + j] = run;
            run += c;
        }
    __syncthreads();
    return total;
}

__device__ void build_matched_lists(const SolveParams& prm, int pair, State& st, double* sortbuf, Feat& f, uint16_t* midx_p,
                                    uint16_t* midx_l, int& n1p, int& n1l, size_t& out_p0, size_t& out_l0, long long& t_ph,
                                    const RecordSink& rs) {
    const int tid = threadIdx.x, nth = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nth >> 5;
    const PlConfig& cfg = prm.cfg;
    if (prm.mode == 0) {
        // ---- A. finish the matching: ratio test, mutual filter -> m12 (global) ----
        const MatchProblem pp = prm.problems[2 * pair], pl = prm.problems[2 * pair + 1];
        match_finalize_block(pp, reinterpret_cast<uint16_t*>(sortbuf));
        __syncthreads();
        match_finalize_block(pl, reinterpret_cast<uint16_t*>(sortbuf));
        __syncthreads();
        if (tid == 0) { st.tc[0] += clock64() - t_ph; }
        t_ph = clock64();

        // ---- B. f2fTracking glue: ordered compaction of the matched features into SoA (and, streamed solver, fp32 records) ----
        const FrameDev& P = prm.prev;
        const FrameDev& C = prm.curr;
        int* cc = reinterpret_cast<int*>(sortbuf);
        const int a0 = P.pt_off[pair], b0 = C.pt_off[pair];
        n1p = P.pt_off[pair + 1] - a0;
        out_p0 = (size_t)a0;
        {
            const int np = compaction_plan(st, pp.m12, n1p, cc);
            const int nch = (n1p + 31) >> 5;
            for (int ch = warp; ch < nch; ch += nw) {
                const int i = ch * 32 + lane;
                const int i2 = (i < n1p) ? pp.m12[i] : -1;
                const unsigned bal = __ballot_sync(FULL_MASK, i2 >= 0);
                if (i2 >= 0) {
                    const int k = cc[ch] + __popc(bal & ((1u << lane) - 1u));
                    const double* p3 = P.pt_P + 3 * (size_t)(a0 + i);
                    const double* o2 = C.pt_pl + 2 * (size_t)(b0 + i2);    // pl_obs = curr pl (:148)
                    const double x = p3[0], y = p3[1], z = p3[2], u = o2[0], v = o2[1];
                    const double pss = sqrt(P.pt_sigma2[a0 + i]);          // PointFeature::safeCopy keeps sigma2
                    f.Px[k] = x; f.Py[k] = y; f.Pz[k] = z;
                    f.pu[k] = u; f.pv[k] = v;
                    f.pss[k] = pss;
                    f.inl_p[k] = 1;
                    midx_p[k] = (uint16_t)i;
                    if (rs.on) sink_point(rs, k, np, x, y, z, u, v, pss, true);
                }
            }
            f.np = np;
            __syncthreads();                 // cc is reused by the lines
        }
        const int c0 = P.ls_off[pair], d0 = C.ls_off[pair];
        n1l = P.ls_off[pair + 1] - c0;
        out_l0 = (size_t)c0;
        {
            const int nl = compaction_plan(st, pl.m12, n1l, cc);
            const int nch = (n1l + 31) >> 5;
            for (int ch = warp; ch < nch; ch += nw) {
                const int i = ch * 32 + lane;
                const int i2 = (i < n1l) ? pl.m12[i] : -1;
                const unsigned bal = __ballot_sync(FULL_MASK, i2 >= 0);
                if (i2 >= 0) {
                    const int k = cc[ch] + __popc(bal & ((1u << lane) - 1u));
                    const size_t a = (size_t)(c0 + i);
                    const double sx = P.ls_sP[3 * a], sy = P.ls_sP[3 * a + 1], sz = P.ls_sP[3 * a + 2];
                    const double ex = P.ls_eP[3 * a], ey = P.ls_eP[3 * a + 1], ez = P.ls_eP[3 * a + 2];
                    const double* le = C.ls_le + 3 * (size_t)(d0 + i2);    // le_obs = curr le (:175)
                    const double l0 = le[0], l1 = le[1], l2 = le[2];
                    double oa, ob, oc;
                    overlap_coeffs(P.ls_spl[2 * a], P.ls_spl[2 * a + 1], P.ls_epl[2 * a], P.ls_epl[2 * a + 1], oa, ob, oc);
                    // LineFeature::safeCopy -> ctor re-applies the level rule (src/stereoFeatures.cpp:117-135):
                    // sigma2' = 1 / (sigma2 * lsdScale^level)^2
                    double s2 = P.ls_sigma2[a];
                    const int level = P.ls_level ? P.ls_level[a] : 0;
                    for (int l = 0; l < level; l++) s2 *= cfg.lsd_scale;
                    const double lss = sqrt(1.0 / (s2 * s2));
                    f.sX[k] = sx; f.sY[k] = sy; f.sZ[k] = sz;
                    f.eX[k] = ex; f.eY[k] = ey; f.eZ[k] = ez;
                    f.l0[k] = l0; f.l1[k] = l1; f.l2[k] = l2;
                    f.oa[k] = oa; f.ob[k] = ob; f.oc[k] = oc;
                    f.lss[k] = lss;
                    f.inl_l[k] = 1;
                    midx_l[k] = (uint16_t)i;
                    if (rs.on) sink_line(rs, k, nl, sx, sy, sz, ex, ey, ez, l0, l1, l2, oa, ob, oc, lss, true);
                }
            }
            f.nl = nl;
        }
        if (tid == 0) {
            st.n_inl_p = f.np;   // f2fTracking: n_inliers_* = list sizes (:126-128)
            st.n_inl_l = f.nl;
        }
    } else {
        // ---- explicit matched lists ----
        const MatchedDev& M = prm.matched;
        const int a0 = M.pt_off[pair], c0 = M.ls_off[pair];
        n1p = f.np = M.pt_off[pair + 1] - a0;
        n1l = f.nl = M.ls_off[pair + 1] - c0;
        out_p0 = (size_t)a0;
        out_l0 = (size_t)c0;
        for (int i = tid; i < f.np; i += nth) {
            const size_t a = (size_t)(a0 + i);
            const double x = M.pt_P[3 * a], y = M.pt_P[3 * a + 1], z = M.pt_P[3 * a + 2];
            const double u = M.pt_pl_obs[2 * a], v = M.pt_pl_obs[2 * a + 1], pss = sqrt(M.pt_sigma2[a]);
            const bool inl = M.pt_inlier ? (M.pt_inlier[a] != 0) : true;
            f.Px[i] = x; f.Py[i] = y; f.Pz[i] = z;
            f.pu[i] = u; f.pv[i] = v;
            f.pss[i] = pss;
            f.inl_p[i] = inl ? 1 : 0;
            if (rs.on) sink_point(rs, i, f.np, x, y, z, u, v, pss, inl);
        }
        for (int i = tid; i < f.nl; i += nth) {
            const size_t a = (size_t)(c0 + i);
            const double sx = M.ls_sP[3 * a], sy = M.ls_sP[3 * a + 1], sz = M.ls_sP[3 * a + 2];
            const double ex = M.ls_eP[3 * a], ey = M.ls_eP[3 * a + 1], ez = M.ls_eP[3 * a + 2];
            const double l0 = M.ls_le_obs[3 * a], l1 = M.ls_le_obs[3 * a + 1], l2 = M.ls_le_obs[3 * a + 2];
            double oa, ob, oc;
            overlap_coeffs(M.ls_spl[2 * a], M.ls_spl[2 * a + 1], M.ls_epl[2 * a], M.ls_epl[2 * a + 1], oa, ob, oc);
            const double lss = sqrt(M.ls_sigma2[a]);
            const bool inl = M.ls_inlier ? (M.ls_inlier[a] != 0) : true;
            f.sX[i] = sx; f.sY[i] = sy; f.sZ[i] = sz;
            f.eX[i] = ex; f.eY[i] = ey; f.eZ[i] = ez;
            f.l0[i] = l0; f.l1[i] = l1; f.l2[i] = l2;
            f.oa[i] = oa; f.ob[i] = ob; f.oc[i] = oc;
            f.lss[i] = lss;
            f.inl_l[i] = inl ? 1 : 0;
            if (rs.on) sink_line(rs, i, f.nl, sx, sy, sz, ex, ey, ez, l0, l1, l2, oa, ob, oc, lss, inl);
        }
        // the reference sets n_inliers from the list sizes; explicit flags only matter to the evaluator
        if (tid == 0) {
            st.n_inl_p = f.np;
            st.n_inl_l = f.nl;
        }
    }
}

__global__ void __launch_bounds__(K2_THREADS, 1) track_solve_kernel(const SolveParams prm) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int tid = threadIdx.x, nth = blockDim.x, lane = tid & 31, warp = tid >> 5;
    const int pair = prm.first_pair + blockIdx.x;
    if (prm.only_if && !prm.only_if[blockIdx.x]) return;   // streamed path: only the problems it handed back

    // ---- carve shared memory ----
    State& st = *reinterpret_cast<State*>(smem);
    size_t off = align_up(sizeof(State), 16);
    double* sortbuf = reinterpret_cast<double*>(smem + off);
    off += (size_t)prm.sort_cap * sizeof(double);
    Feat f;
    f.inl_p = smem + off;  off += align_up((size_t)prm.cap_pt, 16);
    f.inl_l = smem + off;  off += align_up((size_t)prm.cap_ls, 16);
    uint16_t* midx_p = reinterpret_cast<uint16_t*>(smem + off);  off += align_up((size_t)prm.cap_pt * 2, 16);
    uint16_t* midx_l = reinterpret_cast<uint16_t*>(smem + off);  off += align_up((size_t)prm.cap_ls * 2, 16);
    double* fb = prm.feat_in_smem ? reinterpret_cast<double*>(smem + off)
                                  : prm.feat_scratch + (size_t)blockIdx.x * prm.feat_scratch_stride;
    {
        const int cp = prm.cap_pt, cl = prm.cap_ls;
        f.Px = fb; f.Py = fb + cp; f.Pz = fb + 2 * cp; f.pu = fb + 3 * cp; f.pv = fb + 4 * cp; f.pss = fb + 5 * cp;
        double* lb = fb + PT_ARRAYS * (size_t)cp;
        f.sX = lb; f.sY = lb + cl; f.sZ = lb + 2 * cl; f.eX = lb + 3 * cl; f.eY = lb + 4 * cl; f.eZ = lb + 5 * cl;
        f.l0 = lb + 6 * cl; f.l1 = lb + 7 * cl; f.l2 = lb + 8 * cl; f.oa = lb + 9 * cl; f.ob = lb + 10 * cl;
        f.oc = lb + 11 * cl; f.lss = lb + 12 * cl;
    }
    const PlConfig& cfg = prm.cfg;
    const Cam cam = {prm.cam.fx, prm.cam.fy, prm.cam.cx, prm.cam.cy};

    if (tid == 0)
        for (int i = 0; i < 8; i++) st.tc[i] = 0;
    long long t_ph = clock64();
    int n1p = 0, n1l = 0;        // prev-frame feature counts (mode 0) / list lengths (mode 1)
    size_t out_p0 = 0, out_l0 = 0;   // where this pair's inlier flags start

    {
        RecordSink none;
        none.on = false;
        build_matched_lists(prm, pair, st, sortbuf, f, midx_p, midx_l, n1p, n1l, out_p0, out_l0, t_ph, none);
    }
    __syncthreads();
    if (tid == 0) { st.tc[1] += clock64() - t_ph; }

    // ---- C. optimizePose (:307-392) ----
    const PlPrior* prior = prm.priors ? &prm.priors[pair] : nullptr;
    if (warp == 0) {
        if (lane == 0) {
            st.out.status = PLSTVO_ST_REFINED;
            st.out.iters_stage1 = st.out.iters_stage2 = 0;
            st.err = -1.0;
        }
        for (int i = lane; i < 36; i += 32) st.cov[i] = 0.0;
        bool use_prior = false;
        if (cfg.use_motion_model && prior) {   // :317-324
            if (lane < 16) st.DT0[lane] = prior->DT[lane];
            for (int i = lane; i < 36; i += 32) st.H[i] = prior->DT_cov[i];   // staging for the gate
            __syncwarp();
            use_prior = warp_is_good_solution(st.DT0, st.H, prior->err_norm, nullptr);
            __syncwarp();
        }
        if (lane < 16) {
            const double v = use_prior ? st.DT0[lane] : ((lane % 5 == 0) ? 1.0 : 0.0);
            st.DT0[lane] = v;
            st.DT[lane] = v;
        }
        if (lane == 0) st.ctrl = (st.n_inl_p + st.n_inl_l >= cfg.min_features) ? 1 : 0;
    }
    __syncthreads();
    const bool robust_mode = (cfg.solver_mode != 0);
    if (st.ctrl) {   // block-uniform
        __syncthreads();
        gauss_newton(f, st, sortbuf, cam, cfg, cfg.max_iters, robust_mode);     // stage 1 on DT_ = DT (:335-338)
        if (warp == 0) {
            const long long t_g = clock64();
            const bool ok = warp_is_good_solution(st.DT, st.cov, st.err, nullptr);   // :341
            if (lane == 0) {
                st.out.iters_stage1 = st.evals;
                st.ctrl = ok ? 1 : 0;
                st.tc[4] += clock64() - t_g;
            }
        }
        __syncthreads();
        if (st.ctrl) {
            __syncthreads();
            const long long t_o = clock64();
            remove_outliers(f, st, sortbuf, st.DT, cam, cfg);                     // at the stage-1 pose (:343)
            if (tid < 16) st.DT[tid] = st.DT0[tid];                               // stage 2 restarts from DT (:347)
            if (tid == 0) {
                st.tc[5] += clock64() - t_o;
                st.ctrl = (st.n_inl_p + st.n_inl_l >= cfg.min_features) ? 1 : 0;
            }
            __syncthreads();
            if (st.ctrl) {
                __syncthreads();
                gauss_newton(f, st, sortbuf, cam, cfg, cfg.max_iters_ref, robust_mode);
                if (tid == 0) st.out.iters_stage2 = st.evals;
            } else {
                if (tid < 16) st.DT[tid] = (tid % 5 == 0) ? 1.0 : 0.0;            // :351-355
                if (tid == 0) st.out.status = PLSTVO_ST_FEW_AFTER;
            }
        } else {
            __syncthreads();
            if (tid < 16) st.DT[tid] = st.DT0[tid];
            __syncthreads();
            gauss_newton(f, st, sortbuf, cam, cfg, cfg.max_iters_ref, true);      // fallback (:357-359)
            if (tid == 0) {
                st.out.iters_stage2 = st.evals;
                st.out.status = PLSTVO_ST_ROBUST_FALLBACK;
            }
        }
    } else {
        if (tid < 16) st.DT[tid] = (tid % 5 == 0) ? 1.0 : 0.0;                    // :364-368
        if (tid == 0) st.out.status = PLSTVO_ST_FEW_BEFORE;
    }
    __syncthreads();

    // ---- pose finalisation (:372-391), warp 0 ----
    if (warp == 0) finalize_pose(st, prior, f, lane, prm.phase_cycles ? prm.phase_cycles + (size_t)pair * 8 : nullptr);
    __syncthreads();
    {   // result struct -> HBM, cooperatively (sizeof(PlPoseResult) is a multiple of 8)
        const uint64_t* src = reinterpret_cast<const uint64_t*>(&st.out);
        uint64_t* dst = reinterpret_cast<uint64_t*>(&prm.results[pair]);
        for (int i = tid; i < (int)(sizeof(PlPoseResult) / 8); i += nth) dst[i] = src[i];
    }
    // ---- inlier flags back to the caller's indexing ----
    if (prm.mode == 0) {
        if (prm.inlier_pt) {
            for (int i = tid; i < n1p; i += nth) prm.inlier_pt[out_p0 + i] = 0;
        }
        if (prm.inlier_ls) {
            for (int i = tid; i < n1l; i += nth) prm.inlier_ls[out_l0 + i] = 0;
        }
        __syncthreads();
        if (prm.inlier_pt)
            for (int k = tid; k < f.np; k += nth) prm.inlier_pt[out_p0 + midx_p[k]] = f.inl_p[k];
        if (prm.inlier_ls)
            for (int k = tid; k < f.nl; k += nth) prm.inlier_ls[out_l0 + midx_l[k]] = f.inl_l[k];
    } else {
        if (prm.inlier_pt)
            for (int k = tid; k < f.np; k += nth) prm.inlier_pt[out_p0 + k] = f.inl_p[k];
        if (prm.inlier_ls)
            for (int k = tid; k < f.nl; k += nth) prm.inlier_ls[out_l0 + k] = f.inl_l[k];
    }
}

// test hook: the warp-level 6x6 routines on caller-supplied matrices (one warp per problem)
__global__ void algebra_selftest_kernel(const double* __restrict__ H, const double* __restrict__ g, int n,
                                        double* __restrict__ x, double* __restrict__ lad, double* __restrict__ inv,
                                        double* __restrict__ eig) {
    __shared__ double sH[36], sg[6], sInv[36];
    const int lane = threadIdx.x & 31, p = blockIdx.x;
    if (p >= n) return;
    for (int i = lane; i < 36; i += 32) sH[i] = H[(size_t)p * 36 + i];
    if (lane < 6) sg[lane] = g[(size_t)p * 6 + lane];
    __syncwarp();
    double xs[6], l, w[6];
    warp_qr6_solve<true>(sH, sg, xs, l);
    warp_inv6(sH, sInv);
    warp_eig6_sym(sH, w);
    if (lane < 6) {
        x[(size_t)p * 6 + lane] = sel6(xs, lane);
        eig[(size_t)p * 6 + lane] = sel6(w, lane);
    }
    if (lane == 0) lad[p] = l;
    for (int i = lane; i < 36; i += 32) inv[(size_t)p * 36 + i] = sInv[i];
}

// test hook: the block-wide radix selection on caller-supplied lists (one 256-thread CTA per list, like the outlier pass); mode 0:
// the k-th smallest value, mode 1: the k-th smallest of |x - pivot| rounded to float (the MAD form of src/auxiliar.cpp:399-402)
__global__ void __launch_bounds__(256) select_selftest_kernel(const double* __restrict__ v, const int32_t* __restrict__ off,
                                                              const int32_t* __restrict__ ks, const double* __restrict__ pivot,
                                                              int mode, double* __restrict__ out) {
    extern __shared__ __align__(16) uint8_t smem[];
    State& st = *reinterpret_cast<State*>(smem);
    const SelScratch sel = sel_scratch_at(smem + align_up(sizeof(State), 16));
    const int p = blockIdx.x, a = off[p], n = off[p + 1] - a;
    if (n <= 0) return;
    const double* x = v + a;
    const double piv = pivot ? pivot[p] : 0.0;
    double r;
    if (mode == 0) r = block_select_wide(sel, st, n, ks[p], [&](int i) -> double { return x[i]; });
    else r = block_select_wide(sel, st, n, ks[p], [&](int i) -> double { return (double)fabsf((float)(x[i] - piv)); });
    if (threadIdx.x == 0) out[p] = r;
}

cudaError_t launch_select_selftest(const double* v, const int32_t* off, const int32_t* ks, const double* pivot, int mode, int n_lists,
                                   double* out, cudaStream_t stream) {
    if (n_lists <= 0) return cudaSuccess;
    const size_t smem = align_up(sizeof(State), 16) + sel_scratch_bytes();
    select_selftest_kernel<<<n_lists, 256, smem, stream>>>(v, off, ks, pivot, mode, out);
    return cudaGetLastError();
}

cudaError_t launch_algebra_selftest(const double* H, const double* g, int n, double* x, double* lad, double* inv,
                                    double* eig, cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    algebra_selftest_kernel<<<n, 32, 0, stream>>>(H, g, n, x, lad, inv, eig);
    return cudaGetLastError();
}

// =====================================================================================================================
// Streamed optimizePose: the same algorithm cut into kernels around HBM-bound evaluation sweeps (see common.cuh)
// =====================================================================================================================
namespace {

struct StreamView {           // per-CTA pointers of the streamed kernels: State + sort buffer in shared memory, lists in HBM
    State* st;
    double* sortbuf;
    Feat f;
    uint16_t *midx_p, *midx_l;
    size_t slot_p, slot_l;    // first record slot of this problem
};

__device__ __forceinline__ StreamView stream_view(const SolveParams& prm, const StreamBufs& sb, uint8_t* smem, int pair, int local) {
    StreamView v;
    v.st = reinterpret_cast<State*>(smem);
    v.sortbuf = reinterpret_cast<double*>(smem + align_up(sizeof(State), 16));
    v.slot_p = (size_t)(prm.mode == 0 ? prm.prev.pt_off[pair] : prm.matched.pt_off[pair]);
    v.slot_l = (size_t)(prm.mode == 0 ? prm.prev.ls_off[pair] : prm.matched.ls_off[pair]);
    v.f.inl_p = sb.flag_pt + v.slot_p;
    v.f.inl_l = sb.flag_ls + v.slot_l;
    v.midx_p = sb.midx_pt + v.slot_p;
    v.midx_l = sb.midx_ls + v.slot_l;
    double* fb = prm.feat_scratch + (size_t)local * prm.feat_scratch_stride;
    const int cp = prm.cap_pt, cl = prm.cap_ls;
    Feat& f = v.f;
    f.Px = fb; f.Py = fb + cp; f.Pz = fb + 2 * cp; f.pu = fb + 3 * cp; f.pv = fb + 4 * cp; f.pss = fb + 5 * cp;
    double* lb = fb + PT_ARRAYS * (size_t)cp;
    f.sX = lb; f.sY = lb + cl; f.sZ = lb + 2 * cl; f.eX = lb + 3 * cl; f.eY = lb + 4 * cl; f.eZ = lb + 5 * cl;
    f.l0 = lb + 6 * cl; f.l1 = lb + 7 * cl; f.l2 = lb + 8 * cl; f.oa = lb + 9 * cl; f.ob = lb + 10 * cl;
    f.oc = lb + 11 * cl; f.lss = lb + 12 * cl;
    f.np = f.nl = 0;
    return v;
}


// ---- S1: matching finish + list building + fp32 records + the head of optimizePose (:317-333) ----
// 256-thread CTAs, up to three per SM: list building is a chain of short block-wide steps (see stream_outlier_kernel)
constexpr int SPREP_THREADS = 256;
__host__ __device__ inline size_t stream_prepare_smem(int sort_cap) { return align_up(sizeof(State), 16) + (size_t)sort_cap * sizeof(double); }
__global__ void __launch_bounds__(SPREP_THREADS, 3) stream_prepare_kernel(const SolveParams prm, const StreamBufs sb) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, local = blockIdx.x;
    const int pair = prm.first_pair + local;
    StreamView v = stream_view(prm, sb, smem, pair, local);
    State& st = *v.st;
    if (tid == 0)
        for (int i = 0; i < 8; i++) st.tc[i] = 0;
    long long t_ph = clock64();
    int n1p = 0, n1l = 0;
    size_t out_p0 = 0, out_l0 = 0;
    {
        RecordSink rs;
        rs.on = true;
        rs.pt = sb.rec_pt + 2 * v.slot_p;
        rs.ls = sb.rec_ls + 4 * v.slot_l;
        rs.cam = GsCamD{prm.cam.fx, prm.cam.fy, prm.cam.cx, prm.cam.cy};
        build_matched_lists(prm, pair, st, v.sortbuf, v.f, v.midx_p, v.midx_l, n1p, n1l, out_p0, out_l0, t_ph, rs);
    }
    __syncthreads();
    const PlConfig& cfg = prm.cfg;
    const PlPrior* prior = prm.priors ? &prm.priors[pair] : nullptr;
    StreamCtl& c = sb.ctl[local];
    if (warp == 0) {
        bool use_prior = false;
        if (cfg.use_motion_model && prior) {   // :317-324
            if (lane < 16) st.DT0[lane] = prior->DT[lane];
            for (int i = lane; i < 36; i += 32) st.H[i] = prior->DT_cov[i];
            __syncwarp();
            use_prior = warp_is_good_solution(st.DT0, st.H, prior->err_norm, nullptr);
            __syncwarp();
        }
        if (lane < 16) {
            const double d = use_prior ? st.DT0[lane] : ((lane % 5 == 0) ? 1.0 : 0.0);
            c.DT0[lane] = d;
            sb.DT[(size_t)local * 16 + lane] = d;
        }
        for (int i = lane; i < 36; i += 32) c.cov[i] = 0.0;
        if (lane == 0) {
            const bool enough = v.f.np + v.f.nl >= cfg.min_features;
            c.err = -1.0;
            c.err_prev = 999999999.9;
            c.iters = 0;
            c.phase = 1;
            c.fail_first = 0;
            c.delegate = (cfg.solver_mode != 0) ? 1 : 0;       // the robust main solver stays with K2
            c.done = enough ? 0 : 1;
            c.status = enough ? PLSTVO_ST_REFINED : PLSTVO_ST_FEW_BEFORE;
            c.iters1 = c.iters2 = 0;
            c.n_inl_p = v.f.np;
            c.n_inl_l = v.f.nl;
            c.np = v.f.np;
            c.nl = v.f.nl;
            sb.cnt_pt[local] = v.f.np;
            sb.cnt_ls[local] = v.f.nl;
            sb.active[local] = (enough && !c.delegate) ? 1 : 0;
            if (!enough)                                          // :364-368: DT = I
                for (int i = 0; i < 16; i++) sb.DT[(size_t)local * 16 + i] = (i % 5 == 0) ? 1.0 : 0.0;
        }
    }
}

// e = sum w r^2 and N of optimizeFunctions (:549-694) in fp64 from the fp64 lists, this thread's share (features tid, tid + nth, ...):
// what the streamed loop falls back on when one of its stop tests is too close to call on the fp32-evaluated error.
__device__ void exact_error_partial(const Feat& f, const double* DT, const Cam& cam, double& e_out, double& n_out) {
    const int tid = threadIdx.x, nth = blockDim.x;
    double e = 0.0, n = 0.0;
    for (int i = tid; i < f.np; i += nth) {
        if (!f.inl_p[i]) continue;
        double X, Y, Z, iz, dx, dy;
        const double r = point_residual(f, i, DT, cam, X, Y, Z, iz, dx, dy) * f.pss[i];
        e += r * r * (1.0 / (1.0 + r * r));
        n += 1.0;
    }
    for (int i = tid; i < f.nl; i += nth) {
        if (!f.inl_l[i]) continue;
        LineRes lr;
        const double r = line_residual(f, i, DT, cam, lr) * f.lss[i];
        double w = 1.0 / (1.0 + r * r);
        const double oa = f.oa[i], ob = f.ob[i], oc = f.oc[i];
        w *= overlap_from_lambdas(oa * lr.spu + ob * lr.spv + oc, oa * lr.epu + ob * lr.epv + oc);
        e += r * r * w;
        n += 1.0;
    }
    e_out = e;
    n_out = n;
}

// ---- S2: the whole Gauss-Newton call of one problem inside one persistent CTA, its records streamed from HBM every iteration ----
// gaussNewtonOptimization (:394-431) for the streamed solver.  CTAs (2 per SM) take problems from an atomic queue; per
// iteration the producer lane streams the problem's 16 KB record tiles through a TMA ring (cp.async.bulk + mbarriers), eight
// consumer warps evaluate optimizeFunctions on them (fp32 per feature, folded to fp64 every few tiles, fixed order), warp 0 sums
// the warps, runs the stop tests / 6x6 solve / SE(3) update in double and publishes the new pose.  No grid-wide step between
// iterations: while one CTA of an SM solves its 6x6 system the other keeps the memory pipe busy, so the launch as a whole
// streams at HBM speed.  One launch replaces max_iters x (sweep + reduce + step).
#ifndef GL_FOLD_TILES
#define GL_FOLD_TILES 4
#endif
constexpr int GL_FOLD = GL_FOLD_TILES;
// CTA shape of the GN loop kernel: consumer warps, ring stages, CTAs per SM (three digits).  862 keeps a KITTI-size problem's
// records resident in the ring.  434 (twice the problems in flight per SM, records re-streamed from L2 every iteration) was
// measured: the kernel alone gets faster at C2 (0.262 -> 0.227 ms per 512 problems) but the pass as a whole does not (two solver
// chains already run side by side), and C5's stage 2 gets slower (0.45 -> 0.51 ms).
#ifndef GL_SHAPE
#define GL_SHAPE 862
#endif
constexpr int GL_CWARPS = GL_SHAPE / 100, GL_STAGES = (GL_SHAPE / 10) % 10, GL_MINBLOCKS = GL_SHAPE % 10;
constexpr int GL_CONSUMERS = GL_CWARPS * 32, GL_THREADS = GL_CONSUMERS + 32;
constexpr double GL_ERR_BAND = 2.5e-7;   // relative half-width of the "could go either way" band of the error tests (~10x the noise)
constexpr double GL_INC_BAND = 1e-3;     // the same for the increment-norm test   // tiles between fp32 -> fp64 folds of a thread's accumulators
__global__ void __launch_bounds__(GL_THREADS, GL_MINBLOCKS)
gn_loop_stream_kernel(const PlCamera cam, const PlConfig cfg, const int32_t* __restrict__ pt_off, const int32_t* __restrict__ ls_off,
                      const StreamBufs sb, int n, int max_iters, int* __restrict__ queue, double* __restrict__ feat_scratch,
                      size_t feat_stride, int cap_pt, int cap_ls) {
    extern __shared__ __align__(128) uint8_t ring[];
    __shared__ __align__(8) uint64_t full[GL_STAGES], empty[GL_STAGES];
    __shared__ double red[GL_CWARPS + 1][32], sH[36], sg[8], sDT[16], sDTprev[16], sC[36], s_exact[4];
    __shared__ float sPose[12];
    __shared__ int s_prob, s_stop, s_amb;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        for (int st = 0; st < GL_STAGES; ++st) {
            mbar_init(&full[st], 1);
            mbar_init(&empty[st], GL_CWARPS);
        }
        fence_mbar_init();
    }
    __syncthreads();
    GsPose P;
    P.fx = (float)cam.fx; P.fy = (float)cam.fy; P.cx = (float)cam.cx; P.cy = (float)cam.cy;
    P.h = (float)cfg.homog_th; P.inv_h = 1.f / P.h; P.fx_h = P.fx / P.h;
    uint32_t k = 0;   // tiles through the ring so far: producer and consumers count the same sequence
    for (;;) {
        if (tid == 0) s_prob = atomicAdd(queue, 1);
        __syncthreads();
        const int p = s_prob;
        if (p >= n) break;
        const bool live = sb.active[p] != 0;
        __syncthreads();                       // s_prob may be rewritten only after everyone has read it
        if (!live) continue;
        StreamCtl& c = sb.ctl[p];
        const int np = sb.cnt_pt[p], nl = sb.cnt_ls[p], p0 = pt_off[p], l0 = ls_off[p];
        const int ptiles = (np + GS_PT_TILE - 1) / GS_PT_TILE, n_tiles = ptiles + (nl + GS_LS_TILE - 1) / GS_LS_TILE;
        // a problem whose records fit the ring (KITTI-size: 4 point tiles + 2 line tiles) is loaded ONCE per GN call and
        // re-evaluated from shared memory; longer lists stream through the ring every iteration
        const bool resident = n_tiles <= GL_STAGES;
        if (tid < 16) sDT[tid] = sb.DT[(size_t)p * 16 + tid];
        if (tid < 12) sPose[tid] = gs_pose_entry(sb.DT[(size_t)p * 16 + tid], tid);
        double err_prev = c.err_prev, err = 0.0;   // warp 0's copies are the authoritative ones
        int it = 0;
        bool fail_first = false, delegated = false;
        __syncthreads();
        for (;; ++it) {
            if (warp == GL_CWARPS) {           // ---- producer ----
                if (lane == 0 && (!resident || it == 0)) {
                    for (int t = 0; t < n_tiles; ++t) {
                        const uint32_t kk = k + t, st = kk % GL_STAGES;
                        if (kk >= GL_STAGES) mbar_wait(&empty[st], ((kk / GL_STAGES) - 1) & 1);
                        const void* src;
                        uint32_t bytes;
                        if (t < ptiles) {
                            src = sb.rec_pt + 2 * (size_t)(p0 + t * GS_PT_TILE);
                            bytes = (uint32_t)min(GS_PT_TILE, np - t * GS_PT_TILE) * 32u;
                        } else {
                            const int f0 = (t - ptiles) * GS_LS_TILE;
                            src = sb.rec_ls + 4 * (size_t)(l0 + f0);
                            bytes = (uint32_t)min(GS_LS_TILE, nl - f0) * 64u;
                        }
                        mbar_arrive_expect_tx(&full[st], bytes);
                        bulk_g2s(ring + (size_t)st * GS_STAGE_BYTES, src, bytes, &full[st]);
                    }
                }
            } else {                           // ---- consumers ----
#pragma unroll
                for (int i = 0; i < 12; i++) P.r[i] = sPose[i];
                GsAccPacked acc;
                acc.clear();
                double run = 0.0;              // lane L: this warp's fp64 total of accumulator L so far
                for (int t = 0; t < n_tiles; ++t) {
                    const uint32_t kk = k + t, st = kk % GL_STAGES;
                    if (!resident || it == 0) mbar_wait(&full[st], (kk / GL_STAGES) & 1);
                    const float4* sr = reinterpret_cast<const float4*>(ring + (size_t)st * GS_STAGE_BYTES);
                    if (t < ptiles) {
                        const int cnt = min(GS_PT_TILE, np - t * GS_PT_TILE);
#pragma unroll
                        for (int h = 0; h < GS_PT_TILE / GL_CONSUMERS; ++h) {
                            const int idx = tid + h * GL_CONSUMERS;
                            const bool lv = idx < cnt;
                            const int ii = lv ? idx : 0;
                            const float4 a = sr[ii], b = sr[cnt + ii];
                            gs_point(P, a, b, lv && b.z != 0.f, acc);
                        }
                    } else {
                        const int cnt = min(GS_LS_TILE, nl - (t - ptiles) * GS_LS_TILE);
#pragma unroll
                        for (int h = 0; h < GS_LS_TILE / GL_CONSUMERS; ++h) {
                            const int idx = tid + h * GL_CONSUMERS;
                            const bool lv = idx < cnt;
                            const int ii = lv ? idx : 0;
                            const float4 a = sr[ii], b = sr[cnt + ii], cc = sr[2 * cnt + ii], d = sr[3 * cnt + ii];
                            gs_line(P, a, b, cc, d, lv && b.w != 0.f, acc);
                        }
                    }
                    __syncwarp();
                    if (lane == 0 && !resident) mbar_arrive(&empty[st]);
                    if ((t % GL_FOLD) == GL_FOLD - 1 || t == n_tiles - 1) {   // fp32 partials -> fp64, fixed order
                        float v[32];
                        acc.unpack(v);
#pragma unroll
                        for (int i = GS_NACC; i < 32; i++) v[i] = 0.f;
#pragma unroll
                        for (int off = 16; off >= 1; off >>= 1) {
                            const bool up = (lane & off) != 0;
#pragma unroll
                            for (int i = 0; i < off; i++) {
                                const float mine = up ? v[i + off] : v[i];
                                const float send = up ? v[i] : v[i + off];
                                v[i] = mine + __shfl_xor_sync(FULL_MASK, send, off);
                            }
                        }
                        run += (double)v[0];
                        acc.clear();
                    }
                }
                red[warp][lane] = run;
            }
            __syncthreads();
            if (warp == 0) {                   // ---- the loop body of :404-427 on the summed normal equations ----
                double sum = 0.0;
#pragma unroll
                for (int w = 0; w < GL_CWARPS; w++) sum += red[w][lane];
                const double cnt = __shfl_sync(FULL_MASK, sum, 28), esum = __shfl_sync(FULL_MASK, sum, 27);
                if (lane < 21) {
                    int i = 0, q = lane;
                    while (q >= 6 - i) { q -= 6 - i; i++; }
                    const int j = i + q;
                    sH[i * 6 + j] = sum;
                    sH[j * 6 + i] = sum;
                } else if (lane < 27) {
                    sg[lane - 21] = sum;
                }
                __syncwarp();
                err = esum / cnt;              // e /= (N_l + N_p)  (:692)
                // The stop tests compare fp32-evaluated errors (relative noise ~3e-8 with the delta-form residuals).  Whether the
                // loop stops HERE — before this iteration's increment — hinges on one number: err - err_prev against
                // -min_error_change (a rise of the error stops it as well), and on err against min_error.  When that number is
                // inside the noise band of the evaluation the reference could have gone either way: the two errors are then
                // formed again in fp64 from the fp64 lists, by the whole CTA, and the tests run on those.
                const double band = GL_ERR_BAND * fabs(err);
                const bool close_call = fabs((err - err_prev) + cfg.min_error_change) <= band || fabs(err - cfg.min_error) <= band;
                if (lane == 0) s_amb = close_call ? 1 : 0;
            }
            __syncthreads();
            if (s_amb) {                       // block-uniform, rare (about one problem in a hundred, once)
                Feat f;
                {
                    double* fb = feat_scratch + (size_t)p * feat_stride;
                    const int cp = cap_pt, cl = cap_ls;
                    f.Px = fb; f.Py = fb + cp; f.Pz = fb + 2 * cp; f.pu = fb + 3 * cp; f.pv = fb + 4 * cp; f.pss = fb + 5 * cp;
                    double* lb = fb + PT_ARRAYS * (size_t)cp;
                    f.sX = lb; f.sY = lb + cl; f.sZ = lb + 2 * cl; f.eX = lb + 3 * cl; f.eY = lb + 4 * cl; f.eZ = lb + 5 * cl;
                    f.l0 = lb + 6 * cl; f.l1 = lb + 7 * cl; f.l2 = lb + 8 * cl; f.oa = lb + 9 * cl; f.ob = lb + 10 * cl;
                    f.oc = lb + 11 * cl; f.lss = lb + 12 * cl;
                    f.inl_p = sb.flag_pt + p0;
                    f.inl_l = sb.flag_ls + l0;
                    f.np = np;
                    f.nl = nl;
                }
                const Cam camd = {cam.fx, cam.fy, cam.cx, cam.cy};
                double v[4];
                exact_error_partial(f, sDT, camd, v[0], v[1]);
                exact_error_partial(f, sDTprev, camd, v[2], v[3]);   // (unused when it == 0: there is no previous pose yet)
#pragma unroll
                for (int q = 0; q < 4; q++)
#pragma unroll
                    for (int o = 16; o; o >>= 1) v[q] += shfl_xor(v[q], o);
                if (lane < 4) red[warp][lane] = (lane == 0) ? v[0] : (lane == 1) ? v[1] : (lane == 2) ? v[2] : v[3];
                __syncthreads();
                if (tid < 4) {
                    double t = 0.0;
                    for (int w = 0; w <= GL_CWARPS; w++) t += red[w][tid];
                    s_exact[tid] = t;
                }
                __syncthreads();
            }
            if (warp == 0) {
                bool stop = false, ambiguous = false;
                if (s_amb) {
                    err = s_exact[0] / s_exact[1];
                    if (it > 0) err_prev = s_exact[2] / s_exact[3];
                }
                if (err > err_prev) {                                             // :405-410
                    stop = true;
                    fail_first = (it == 0);
                } else if ((err < cfg.min_error) || fabs(err - err_prev) < cfg.min_error_change) {   // :412-415
                    stop = true;
                } else {
                    double inc[6], lad;
                    if (!warp_chol6_solve(sH, sg, inc)) warp_qr6_solve<false>(sH, sg, inc, lad);   // :417-418
                    if (lane < 16) sDTprev[lane] = sDT[lane];
                    __syncwarp();
                    apply_increment(sDT, inc, lane);                              // :419
                    if (lane < 12) sPose[lane] = gs_pose_entry(sDT[lane], lane);
                    const double nt = sqrt(inc[0] * inc[0] + inc[1] * inc[1] + inc[2] * inc[2]);
                    const double nr = sqrt(inc[3] * inc[3] + inc[4] * inc[4] + inc[5] * inc[5]);
                    if (nt < cfg.min_error_change && nr < cfg.min_error_change) stop = true;   // :421-424
                    const double ib = GL_INC_BAND * cfg.min_error_change;
                    // an increment whose norm sits on its threshold: the one test left to the fp64 kernel (K2 retraces the problem)
                    ambiguous = (fabs(nt - cfg.min_error_change) <= ib && nr < cfg.min_error_change + ib) ||
                                (fabs(nr - cfg.min_error_change) <= ib && nt < cfg.min_error_change + ib);
                    err_prev = err;
                }
                if (ambiguous) {
                    stop = true;
                    delegated = true;
                }
                if (!stop && it + 1 >= max_iters) stop = true;                    // the for loop runs out
                if (lane == 0) s_stop = stop ? 1 : 0;
            }
            __syncthreads();
            const int stop = s_stop;
            __syncthreads();
            if (!resident) k += n_tiles;       // a streamed iteration used n_tiles ring slots
            if (stop) break;
        }
        if (resident) {                        // the records sat in the ring for the whole call: hand the stages back now
            if (warp < GL_CWARPS && lane == 0)
                for (int t = 0; t < n_tiles; ++t) mbar_arrive(&empty[(k + t) % GL_STAGES]);
            k += n_tiles;
        }
        if (warp == 0) {                       // :429-430 and the state the next kernels read
            if (!fail_first && !delegated) {
                warp_inv6(sH, sC);
                __syncwarp();
                for (int i = lane; i < 36; i += 32) c.cov[i] = sC[i];
            }
            if (lane < 16) sb.DT[(size_t)p * 16 + lane] = sDT[lane];
            if (lane == 0) {
                if (delegated) c.delegate = 1;
                c.err = fail_first ? -1.0 : err;
                c.fail_first = fail_first ? 1 : 0;
                c.iters = it + 1;
                c.err_prev = err_prev;
                sb.active[p] = 0;
            }
        }
        __syncthreads();
    }
}

// ---- S3: gate of stage 1 (:341), removeOutliers at the stage-1 pose (:343), restart for stage 2 (:345-355) ----
// 256-thread CTAs, several per SM (the work is a chain of short block-wide steps: more problems in flight beat wider CTAs).
// Warp 0 runs the gate while the other warps already form the residuals it will (almost always) let through.
constexpr int SO_THREADS = 256;
__host__ __device__ inline size_t stream_outlier_smem(int sort_cap) {
    return align_up(sizeof(State), 16) + (size_t)sort_cap * sizeof(double) + sel_scratch_bytes();
}
__global__ void __launch_bounds__(SO_THREADS, 3) stream_outlier_kernel(const SolveParams prm, const StreamBufs sb) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, local = blockIdx.x;
    const int pair = prm.first_pair + local;
    StreamCtl& c = sb.ctl[local];
    if (c.done || c.delegate) return;
    StreamView v = stream_view(prm, sb, smem, pair, local);
    State& st = *v.st;
    const SelScratch sel = sel_scratch_at(smem + align_up(sizeof(State), 16) + (size_t)prm.sort_cap * sizeof(double));
    v.f.np = c.np;
    v.f.nl = c.nl;
    const PlConfig& cfg = prm.cfg;
    const Cam cam = {prm.cam.fx, prm.cam.fy, prm.cam.cx, prm.cam.cy};
    // the lists live in HBM here: every residual is formed ONCE (same fp64 arithmetic as K2's), straight into shared memory
    if (warp == 0) {
        if (lane == 0) {
            for (int i = 0; i < 8; i++) st.tc[i] = 0;
            st.n_inl_p = c.n_inl_p;
            st.n_inl_l = c.n_inl_l;
        }
        if (lane < 16) st.DT[lane] = sb.DT[(size_t)local * 16 + lane];
        for (int i = lane; i < 36; i += 32) st.cov[i] = c.cov[i];
        __syncwarp();
        const bool ok = warp_is_good_solution(st.DT, st.cov, c.err, nullptr);
        if (lane == 0) st.ctrl = ok ? 1 : 0;
    }
    double DTr[12];                           // pose in registers: the residual loops are pure streaming arithmetic
#pragma unroll
    for (int i = 0; i < 12; i++) DTr[i] = sb.DT[(size_t)local * 16 + i];
    const Feat& f = v.f;
    auto res_pt = [&](int i) -> double {
        double X, Y, Z, iz, dx, dy;
        return point_residual(f, i, DTr, cam, X, Y, Z, iz, dx, dy) * f.pss[i];
    };
    auto res_ls = [&](int i) -> double {
        LineRes r;
        return line_residual(f, i, DTr, cam, r) * f.lss[i];
    };
    const bool pts = cfg.has_points && f.np > 0;
    if (warp != 0 && pts) {                   // the other warps already form the point residuals the gate will (almost always) let through
        const int wt = tid - 32, nwt = SO_THREADS - 32;
#pragma unroll 4
        for (int i = wt; i < f.np; i += nwt) v.sortbuf[i] = res_pt(i);
    }
    __syncthreads();
    if (!st.ctrl) {                     // stage 1 rejected: the robust fallback (:357-359) is K2's job
        if (tid == 0) c.delegate = 1;
        return;
    }
    float4* rec_p = sb.rec_pt + 2 * v.slot_p;
    float4* rec_l = sb.rec_ls + 4 * v.slot_l;
    const int np = f.np, nl = f.nl;
    remove_outliers_select(
        f, st, v.sortbuf, sel, cfg, pts, res_pt, res_ls,
        [&](int j) {   // the inlier flag inside the fp32 record (gn_stream.cuh "records")
            const int t = j / GS_PT_TILE, r = j % GS_PT_TILE, cnt = min(GS_PT_TILE, np - t * GS_PT_TILE);
            reinterpret_cast<float*>(rec_p + 2 * (size_t)t * GS_PT_TILE + cnt + r)[2] = 0.f;
        },
        [&](int j) {
            const int t = j / GS_LS_TILE, r = j % GS_LS_TILE, cnt = min(GS_LS_TILE, nl - t * GS_LS_TILE);
            reinterpret_cast<float*>(rec_l + 4 * (size_t)t * GS_LS_TILE + cnt + r)[3] = 0.f;
        });
    __syncthreads();
    if (tid == 0) {
        c.iters1 = c.iters;
        c.n_inl_p = st.n_inl_p;
        c.n_inl_l = st.n_inl_l;
        if (st.n_inl_p + st.n_inl_l >= cfg.min_features) {   // stage 2 restarts from the INITIAL pose (:347)
            c.phase = 2;
            c.iters = 0;
            c.err_prev = 999999999.9;
            sb.active[local] = 1;
            for (int i = 0; i < 16; i++) sb.DT[(size_t)local * 16 + i] = c.DT0[i];
        } else {                                             // :351-355
            c.status = PLSTVO_ST_FEW_AFTER;
            c.done = 1;
            for (int i = 0; i < 16; i++) sb.DT[(size_t)local * 16 + i] = (i % 5 == 0) ? 1.0 : 0.0;
        }
    }
}

// ---- S4: finalisation (:372-391), result record, inlier flags in the caller's indexing ----
__global__ void __launch_bounds__(256) stream_finalize_kernel(const SolveParams prm, const StreamBufs sb, int32_t* only_if) {
    __shared__ State st;
    const int tid = threadIdx.x, nth = blockDim.x, lane = tid & 31, warp = tid >> 5, local = blockIdx.x;
    const int pair = prm.first_pair + local;
    StreamCtl& c = sb.ctl[local];
    if (tid == 0) only_if[local] = c.delegate;
    if (c.delegate) return;
    Feat f;
    f.np = c.np;
    f.nl = c.nl;
    const size_t slot_p = (size_t)(prm.mode == 0 ? prm.prev.pt_off[pair] : prm.matched.pt_off[pair]);
    const size_t slot_l = (size_t)(prm.mode == 0 ? prm.prev.ls_off[pair] : prm.matched.ls_off[pair]);
    const int n1p = prm.mode == 0 ? prm.prev.pt_off[pair + 1] - (int)slot_p : c.np;
    const int n1l = prm.mode == 0 ? prm.prev.ls_off[pair + 1] - (int)slot_l : c.nl;
    const PlPrior* prior = prm.priors ? &prm.priors[pair] : nullptr;
    if (warp == 0) {
        if (lane < 16) st.DT[lane] = sb.DT[(size_t)local * 16 + lane];
        for (int i = lane; i < 36; i += 32) st.cov[i] = c.cov[i];
        if (lane == 0) {
            for (int i = 0; i < 8; i++) st.tc[i] = 0;
            st.err = c.done ? -1.0 : c.err;
            st.n_inl_p = c.n_inl_p;
            st.n_inl_l = c.n_inl_l;
            st.out.status = c.status;
            st.out.iters_stage1 = (c.phase == 2 || c.done) ? c.iters1 : c.iters;
            st.out.iters_stage2 = (c.phase == 2) ? c.iters : 0;
        }
        __syncwarp();
        finalize_pose(st, prior, f, lane, nullptr);
    }
    __syncthreads();
    {
        const uint64_t* src = reinterpret_cast<const uint64_t*>(&st.out);
        uint64_t* dst = reinterpret_cast<uint64_t*>(&prm.results[pair]);
        for (int i = tid; i < (int)(sizeof(PlPoseResult) / 8); i += nth) dst[i] = src[i];
    }
    const uint8_t* fp = sb.flag_pt + slot_p;
    const uint8_t* fl = sb.flag_ls + slot_l;
    if (prm.mode == 0) {
        if (prm.inlier_pt)
            for (int i = tid; i < n1p; i += nth) prm.inlier_pt[slot_p + i] = 0;
        if (prm.inlier_ls)
            for (int i = tid; i < n1l; i += nth) prm.inlier_ls[slot_l + i] = 0;
        __syncthreads();
        if (prm.inlier_pt)
            for (int k = tid; k < c.np; k += nth) prm.inlier_pt[slot_p + sb.midx_pt[slot_p + k]] = fp[k];
        if (prm.inlier_ls)
            for (int k = tid; k < c.nl; k += nth) prm.inlier_ls[slot_l + sb.midx_ls[slot_l + k]] = fl[k];
    } else {
        if (prm.inlier_pt)
            for (int k = tid; k < c.np; k += nth) prm.inlier_pt[slot_p + k] = fp[k];
        if (prm.inlier_ls)
            for (int k = tid; k < c.nl; k += nth) prm.inlier_ls[slot_l + k] = fl[k];
    }
}

}  // namespace

cudaError_t launch_stream_solve(const SolveParams& prm_in, int n_pairs, const StreamBufs& sb, cudaStream_t stream, int* launches,
                                cudaEvent_t* marks) {
    if (n_pairs <= 0) return cudaSuccess;
    SolveParams prm = prm_in;
    prm.feat_in_smem = 0;
    prm.only_if = nullptr;
    static size_t conf_a[64] = {}, conf_b[64] = {};
    const size_t smem_prep = stream_prepare_smem(prm.sort_cap);
    cudaError_t e = ensure_dynamic_smem(reinterpret_cast<const void*>(stream_prepare_kernel), smem_prep, conf_a);
    if (e != cudaSuccess) return e;
    const size_t smem_out = stream_outlier_smem(prm.sort_cap);
    e = ensure_dynamic_smem(reinterpret_cast<const void*>(stream_outlier_kernel), smem_out, conf_b);
    if (e != cudaSuccess) return e;
    int nl = 0;
    stream_prepare_kernel<<<n_pairs, SPREP_THREADS, smem_prep, stream>>>(prm, sb);
    ++nl;
    // instrumentation (optional): lists built | GN stage 1 done | outlier pass done | GN stage 2 done
    if (marks) cudaEventRecord(marks[0], stream);
    const int32_t* off_p = prm.mode == 0 ? prm.prev.pt_off + prm.first_pair : prm.matched.pt_off + prm.first_pair;
    const int32_t* off_l = prm.mode == 0 ? prm.prev.ls_off + prm.first_pair : prm.matched.ls_off + prm.first_pair;
    static size_t conf_c[64] = {};
    const size_t ring = (size_t)GL_STAGES * GS_STAGE_BYTES;
    e = ensure_dynamic_smem(reinterpret_cast<const void*>(gn_loop_stream_kernel), ring, conf_c);
    if (e != cudaSuccess) return e;
    int gn_calls = 0;
    auto gn = [&](int max_iters) -> cudaError_t {   // one GN call = one launch: persistent CTAs, one problem each at a time
        int* q = sb.queue + (gn_calls++);
        cudaError_t err = cudaMemsetAsync(q, 0, sizeof(int), stream);
        if (err != cudaSuccess) return err;
        const int grid = n_pairs < GL_MINBLOCKS * sb.sm_count ? n_pairs : GL_MINBLOCKS * sb.sm_count;
        gn_loop_stream_kernel<<<grid, GL_THREADS, ring, stream>>>(prm.cam, prm.cfg, off_p, off_l, sb, n_pairs, max_iters, q,
                                                                  prm.feat_scratch, (size_t)prm.feat_scratch_stride, prm.cap_pt, prm.cap_ls);
        nl += 1;
        return cudaGetLastError();
    };
    if ((e = gn(prm.cfg.max_iters)) != cudaSuccess) return e;
    if (marks) cudaEventRecord(marks[1], stream);
    stream_outlier_kernel<<<n_pairs, SO_THREADS, smem_out, stream>>>(prm, sb);
    if (marks) cudaEventRecord(marks[2], stream);
    if ((e = gn(prm.cfg.max_iters_ref)) != cudaSuccess) return e;
    if (marks) cudaEventRecord(marks[3], stream);
    // the activity array doubles as K2's only_if list once the sweeps are over
    stream_finalize_kernel<<<n_pairs, 256, 0, stream>>>(prm, sb, sb.active);
    nl += 2;
    // whatever left the common path: the whole problem again in K2 (global-scratch form)
    SolveParams k2 = prm;
    k2.only_if = sb.active;
    e = launch_track_solve(k2, n_pairs, stream);
    ++nl;
    if (launches) *launches = nl;
    return e != cudaSuccess ? e : cudaGetLastError();
}

cudaError_t launch_track_solve(const SolveParams& prm, int n_pairs, cudaStream_t stream) {
    if (n_pairs <= 0) return cudaSuccess;
    const size_t smem = k2_smem_bytes(prm.cap_pt, prm.cap_ls, prm.sort_cap, prm.feat_in_smem != 0);
    static size_t configured[64] = {};
    cudaError_t e = ensure_dynamic_smem(reinterpret_cast<const void*>(track_solve_kernel), smem, configured);
    if (e != cudaSuccess) return e;
    track_solve_kernel<<<n_pairs, K2_THREADS, smem, stream>>>(prm);
    return cudaGetLastError();
}

}  // namespace plstvo
