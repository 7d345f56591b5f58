// tc_match_test.cu — stand-alone check + timing of the tensor-core matcher (match_tc.cu) against a CPU brute force.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -I stvo_pl_b200/csrc tools/probes/tc_match_test.cu \
//             stvo_pl_b200/csrc/match_tc.cu -o tools/probes/bin/tc_match_test
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <vector>
#include <algorithm>

#include "match_tc.cuh"

using namespace plstvo;

#define CK(x)                                                                                   \
    do {                                                                                        \
        cudaError_t e_ = (x);                                                                   \
        if (e_ != cudaSuccess) {                                                                \
            fprintf(stderr, "CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); \
            exit(2);                                                                            \
        }                                                                                       \
    } while (0)

static int ham(const uint8_t* a, const uint8_t* b) {
    int d = 0;
    for (int i = 0; i < 4; ++i) {
        uint64_t x, y;
        memcpy(&x, a + 8 * i, 8);
        memcpy(&y, b + 8 * i, 8);
        d += __builtin_popcountll(x ^ y);
    }
    return d;
}

struct Prob {
    int n1, n2;
    size_t o1, o2;          // row offsets into the descriptor pools
    size_t e1, e2;          // tile offsets into the expanded pool
    size_t rowp, colp, rowpart, colpart;
};

int main(int argc, char** argv) {
    const int big_pairs = argc > 1 ? atoi(argv[1]) : 64;      // timing batch: pairs of (2000x2000 + 500x500)
    const int tie_mode = argc > 2 ? atoi(argv[2]) : 0;
    const float nnr = 0.75f;
    std::mt19937_64 rng(12345);

    std::vector<std::pair<int, int>> shapes = {{2000, 2000}, {500, 500}, {300, 400}, {130, 257}, {1, 5},   {5, 1},
                                               {2, 2},       {129, 128}, {128, 129}, {257, 511}, {1000, 17}, {17, 1000},
                                               {2000, 2000}, {600, 600}};
    const int n_check = (int)shapes.size();
    for (int p = 0; p < big_pairs; ++p) {
        shapes.push_back({2000, 2000});
        shapes.push_back({500, 500});
    }
    const int P = (int)shapes.size();
    std::vector<Prob> pr(P);
    size_t rows1 = 0, rows2 = 0, tiles = 0, nrowp = 0, ncolp = 0, nrp = 0, ncp = 0;
    for (int p = 0; p < P; ++p) {
        Prob& q = pr[p];
        q.n1 = shapes[p].first;
        q.n2 = shapes[p].second;
        q.o1 = rows1; rows1 += q.n1;
        q.o2 = rows2; rows2 += q.n2;
        const int t1 = (q.n1 + 127) / 128, t2 = (q.n2 + 127) / 128;
        q.e1 = tiles; tiles += t1;
        q.e2 = tiles; tiles += t2;
        q.rowp = nrowp; nrowp += (size_t)((q.n2 + TC_CW - 1) / TC_CW) * q.n1;
        q.colp = ncolp; ncolp += q.n2;
        q.rowpart = nrp; nrp += q.n1;
        q.colpart = ncp; ncp += q.n2;
    }
    std::vector<uint8_t> h1(rows1 * 32), h2(rows2 * 32);
    for (int p = 0; p < P; ++p) {
        const Prob& q = pr[p];
        const bool ties = tie_mode || (p == 12);
        for (size_t i = 0; i < (size_t)q.n1 * 32; ++i) h1[q.o1 * 32 + i] = ties ? ((rng() & 1) ? 0xFF : 0x00) : (uint8_t)rng();
        for (int j = 0; j < q.n2; ++j) {
            uint8_t* d = &h2[(q.o2 + j) * 32];
            if ((rng() % 10) < 7 && q.n1 > 0) {   // noisy copy of a random query row
                const uint8_t* s = &h1[(q.o1 + rng() % q.n1) * 32];
                for (int b = 0; b < 32; ++b) {
                    uint8_t m = 0;
                    for (int k = 0; k < 8; ++k) m |= ((rng() % 10) == 0) << k;
                    d[b] = s[b] ^ (ties ? 0 : m);
                }
            } else {
                for (int b = 0; b < 32; ++b) d[b] = ties ? ((rng() & 1) ? 0xFF : 0x00) : (uint8_t)rng();
            }
        }
    }
    uint8_t *d1, *d2, *ex;
    uint32_t *rowp, *colp;
    uint2 *rowpart, *colpart;
    CK(cudaMalloc(&d1, h1.size() + 32));
    CK(cudaMalloc(&d2, h2.size() + 32));
    CK(cudaMalloc(&ex, tiles * TC_TILE_BYTES));
    CK(cudaMalloc(&rowp, nrowp * 4 + 8));
    CK(cudaMalloc(&colp, ncolp * 4 + 8));
    CK(cudaMalloc(&rowpart, nrp * 8 + 8));
    CK(cudaMalloc(&colpart, ncp * 8 + 8));
    CK(cudaMemcpy(d1, h1.data(), h1.size(), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d2, h2.data(), h2.size(), cudaMemcpyHostToDevice));
    CK(cudaMemset(rowp, 0xAB, nrowp * 4));
    CK(cudaMemset(colp, 0xAB, ncolp * 4));
    CK(cudaMemset(rowpart, 0xCD, nrp * 8));
    CK(cudaMemset(colpart, 0xCD, ncp * 8));

    std::vector<TcSide> sides;
    std::vector<TcProblem> tps(P);
    std::vector<MatchProblem> mps(P);
    std::vector<TcItem> items;
    int max_tiles = 0;
    for (int p = 0; p < P; ++p) {
        const Prob& q = pr[p];
        sides.push_back({d1 + q.o1 * 32, q.n1, ex + q.e1 * TC_TILE_BYTES});
        sides.push_back({d2 + q.o2 * 32, q.n2, ex + q.e2 * TC_TILE_BYTES});
        max_tiles = std::max(max_tiles, std::max((q.n1 + 127) / 128, (q.n2 + 127) / 128));
        tps[p] = {ex + q.e1 * TC_TILE_BYTES, ex + q.e2 * TC_TILE_BYTES, q.n1, q.n2, rowp + q.rowp, colp + q.colp};
        MatchProblem m{};
        m.d1 = d1 + q.o1 * 32; m.d2 = d2 + q.o2 * 32; m.n1 = q.n1; m.n2 = q.n2; m.enabled = 1;
        m.rowpart = rowpart + q.rowpart; m.colpart = colpart + q.colpart; m.nnr = nnr; m.best_lr = 1;
        mps[p] = m;
    }
    // items sorted by decreasing length (query tiles) so the static round-robin stays balanced
    std::vector<int> order(P);
    for (int p = 0; p < P; ++p) order[p] = p;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return pr[a].n1 > pr[b].n1; });
    for (int p : order) {
        const int nyb = (pr[p].n2 + 255) / 256;
        for (int b = 0; b < nyb; ++b) items.push_back({p, b});
    }
    TcSide* dsides; TcProblem* dtps; MatchProblem* dmps; TcItem* ditems; __half* dbg; int* sched;
    CK(cudaMalloc(&sched, 64));
    CK(cudaMemset(sched, 0, 64));
    CK(cudaMalloc(&dsides, sides.size() * sizeof(TcSide)));
    CK(cudaMalloc(&dtps, P * sizeof(TcProblem)));
    CK(cudaMalloc(&dmps, P * sizeof(MatchProblem)));
    CK(cudaMalloc(&ditems, items.size() * sizeof(TcItem)));
    CK(cudaMalloc(&dbg, 128 * 256 * 2));
    CK(cudaMemset(dbg, 0, 128 * 256 * 2));
    CK(cudaMemcpy(dsides, sides.data(), sides.size() * sizeof(TcSide), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dtps, tps.data(), P * sizeof(TcProblem), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dmps, mps.data(), P * sizeof(MatchProblem), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ditems, items.data(), items.size() * sizeof(TcItem), cudaMemcpyHostToDevice));

    int dev = 0, sms = 0;
    CK(cudaGetDevice(&dev));
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    printf("problems %d (checked %d), items %zu, tiles %zu (%.1f MB expanded), SMs %d, smem %zu\n", P, n_check, items.size(),
           tiles, tiles * TC_TILE_BYTES / 1e6, sms, tc_smem_bytes());

    cudaStream_t s;
    CK(cudaStreamCreate(&s));
    CK(launch_tc_expand(dsides, (int)sides.size(), max_tiles, s));
    CK(cudaStreamSynchronize(s));
    printf("expand ok\n"); fflush(stdout);
    CK(launch_tc_hamming(dtps, ditems, (int)items.size(), nullptr, 0, sched, sms, dbg, s));
    CK(cudaStreamSynchronize(s));
    printf("tc ok\n"); fflush(stdout);
    CK(launch_tc_resolve(dmps, dtps, P, 4, s));
    CK(cudaStreamSynchronize(s));
    printf("resolve ok\n"); fflush(stdout);

    // ---- debug tile: first item, first query tile: dots of queries 0..127 against trains 0..255
    {
        std::vector<__half> hd(128 * 256);
        CK(cudaMemcpy(hd.data(), dbg, hd.size() * 2, cudaMemcpyDeviceToHost));
        const int p = items[0].problem, yb = items[0].yblk;
        const Prob& q = pr[p];
        long bad = 0, tot = 0;
        for (int r = 0; r < 128 && r < q.n1; ++r)
            for (int c = 0; c < 256 && yb * 256 + c < q.n2; ++c) {
                const int exp = 256 - 2 * ham(&h1[(q.o1 + r) * 32], &h2[(q.o2 + yb * 256 + c) * 32]);
                const float got = __half2float(hd[r * 256 + c]);
                ++tot;
                if ((float)exp != got) {
                    if (bad < 12) printf("  dot mismatch r=%d c=%d exp=%d got=%g\n", r, c, exp, got);
                    ++bad;
                }
            }
        printf("debug tile (problem %d, yblk %d): %ld / %ld dots wrong\n", p, yb, bad, tot);
    }

    // ---- results vs brute force on the checked problems
    std::vector<uint2> hrow(nrp), hcol(ncp);
    CK(cudaMemcpy(hrow.data(), rowpart, nrp * 8, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(hcol.data(), colpart, ncp * 8, cudaMemcpyDeviceToHost));
    long total_bad = 0;
    const int n_verify = std::min(P, n_check + 4);
    for (int p = 0; p < n_verify; ++p) {
        const Prob& q = pr[p];
        long bad = 0;
        for (int dir = 0; dir < 2; ++dir) {
            const int na = dir ? q.n2 : q.n1, nb = dir ? q.n1 : q.n2;
            const uint8_t* A = dir ? &h2[q.o2 * 32] : &h1[q.o1 * 32];
            const uint8_t* B = dir ? &h1[q.o1 * 32] : &h2[q.o2 * 32];
            const uint2* out = dir ? &hcol[q.colpart] : &hrow[q.rowpart];
            for (int a = 0; a < na; ++a) {
                uint32_t k1 = 0xFFFFFFFFu, k2 = 0xFFFFFFFFu;
                for (int b = 0; b < nb; ++b) {
                    const uint32_t key = ((uint32_t)ham(A + a * 32, B + b * 32) << 16) | (uint32_t)b;
                    if (key < k1) { k2 = k1; k1 = key; } else if (key < k2) k2 = key;
                }
                const uint2 g = out[a];
                bool ok = (g.x >> 16) == (k1 >> 16);
                const bool acc = nb >= 2 && (float)(k1 >> 16) < (float)(k2 >> 16) * nnr;
                // a rejected row / column may carry an upper bound of the second distance instead of the exact one: the
                // decision must agree, the second itself only where the ratio test accepts
                if (nb >= 2) {
                    const bool got_acc = g.y != 0xFFFFFFFFu && (float)(g.x >> 16) < (float)(g.y >> 16) * nnr;
                    ok = ok && got_acc == acc && (!acc || (g.y >> 16) == (k2 >> 16));
                } else {
                    ok = ok && g.y == 0xFFFFFFFFu;
                }
                // column direction: a unique nearest query is left unresolved (index field 0xFFFD): the mutual filter works on
                // the distance alone (match_finalize.cuh)
                const bool unresolved = dir == 1 && (g.x & 0xFFFF) == 0xFFFDu && (k1 >> 16) != (k2 >> 16) && nb <= 0xFE00;
                if (acc && !unresolved) ok = ok && (g.x & 0xFFFF) == (k1 & 0xFFFF);
                if (!ok) {
                    if (bad < 6) printf("  p=%d dir=%d a=%d exp (%u,%u | %u) got (%u,%u | %u,%u) acc=%d\n", p, dir, a, k1 >> 16,
                                        k1 & 0xFFFF, k2 >> 16, g.x >> 16, g.x & 0xFFFF, g.y >> 16, g.y & 0xFFFF, (int)acc);
                    ++bad;
                }
            }
        }
        printf("problem %2d (%4d x %4d): %ld wrong\n", p, q.n1, q.n2, bad);
        total_bad += bad;
    }
    printf("TOTAL wrong: %ld\n", total_bad);

    // ---- timing
    cudaEvent_t e0, e1, e2, e3;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1)); CK(cudaEventCreate(&e2)); CK(cudaEventCreate(&e3));
    float best[3] = {1e9f, 1e9f, 1e9f};
    for (int rep = 0; rep < 10; ++rep) {
        CK(cudaEventRecord(e0, s));
        CK(launch_tc_expand(dsides, (int)sides.size(), max_tiles, s));
        CK(cudaEventRecord(e1, s));
        CK(launch_tc_hamming(dtps, ditems, (int)items.size(), nullptr, 0, sched, sms, nullptr, s));
        CK(cudaEventRecord(e2, s));
        CK(launch_tc_resolve(dmps, dtps, P, 4, s));
        CK(cudaEventRecord(e3, s));
        CK(cudaStreamSynchronize(s));
        float a, b, c;
        CK(cudaEventElapsedTime(&a, e0, e1)); CK(cudaEventElapsedTime(&b, e1, e2)); CK(cudaEventElapsedTime(&c, e2, e3));
        best[0] = std::min(best[0], a); best[1] = std::min(best[1], b); best[2] = std::min(best[2], c);
    }
    double pairs = 0;
    for (int p = 0; p < P; ++p) pairs += (double)pr[p].n1 * pr[p].n2;
    printf("timing (best of 10): expand %.3f ms, tc %.3f ms, resolve %.3f ms; %.3g pair-distances -> %.2f T dist/s (tc only)\n",
           best[0], best[1], best[2], pairs, pairs / best[1] * 1e-9);
    return total_bad ? 1 : 0;
}
