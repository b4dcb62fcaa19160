// Block-band kernels of the 2-D (Kronecker) model as persistent tile-DAG kernels.
//
// P = K1 (x) K2 + G / sigma^2 is block banded with scalar bandwidth w = k (m2 + 1) (reference gpr.py:262); the
// reference factorises it as a DENSE m1 m2 x m1 m2 matrix (tf.linalg.cholesky, gpr.py:293), infeasible at 200 x 200.
//
//   asvgp_kron_factor  <- utils.bands_to_kron_cholesky's Kronecker product, `Kuu + KufKfu / sigma2`,
//                         tf.linalg.cholesky(P), its log-det, triangular_solve(L_P, Kuf_y)     (gpr.py:287-295)
//   asvgp_kron_selinv  <- what TF reverse mode / cholesky_solve extract from P^-1 (gpr.py:307, 319-326): the entries of
//                         P^-1 on the stencil pattern and P^-1 Kuf_y
//   asvgp_kron_terms   <- the scalar contractions of the bound's derivatives and trace(Kuu^-1 KufKfu) (gpr.py:307)
//
// Storage (DESIGN.md §2): the band is cut into NB x NB tiles (NB = 64).  Tile (C, d), d = 0..BW, holds block row C+d of
// block column C as a contiguous column-major 64 x 64 block (32 KB), so one TMA bulk copy (cp.async.bulk, completion
// on an mbarrier) brings a whole operand into shared memory.  BW = floor((w + NB - 1) / NB) sub-diagonals (10 at
// 200 x 200, k = 3); entries of a tile beyond the scalar band are structural zeros and stay exact zeros.
//
// Factorisation = tiled left-looking Cholesky as ONE persistent cooperative kernel: task (R, C) owns tile (R, C),
// subtracts sum_J L(R,J) L(C,J)^T as the operand tiles become final (per-tile release/acquire flags in global
// memory), then either factorises the diagonal tile in registers — right-looking rank-1 sweep that carries L^-1
// along, one barrier per column — or multiplies by the published inverse L(C,C)^-T.  Tasks are dealt round-robin in
// column-major order, which is a topological order of the DAG, so the co-resident CTAs cannot deadlock; the chain of
// diagonal tiles is the critical path, everything else fills the other SMs.  The right-hand side rides along
// (y = L^-1 b), so do log|P| and ||y||^2.
//
// Selected inverse = blocked Takahashi recursion, backwards over block columns, again one persistent kernel:
// Sigma(R,C) = -sum_K Sigma(R,K) Y(K,C), Y = L(K,C) L(C,C)^-1, Sigma(C,C) = L(C,C)^-T L(C,C)^-1 - sum_K Sigma(K,C)^T Y(K,C),
// with the diagonal contributions and the back-substitution x = P^-1 b accumulated by fp64 REDs.  Sigma is kept as
// lower AND upper tiles so that every operand is a plain column-major tile.  No tensor cores: B200's fp64 tensor
// rate equals its fp64 FMA rate (DESIGN.md §4.4).
#include "tile_ops.cuh"
#include "../../include/asvgp_b200.h"

namespace asvgp {


struct TileGeom {
    int m1, m2, K;
    int M;          // m1 * m2
    int nb;         // block rows / columns (M padded to a multiple of NB with unit diagonal)
    int w;          // scalar bandwidth K * m2 + K
    int BW;         // block sub-diagonals
    __host__ __device__ int64_t tile(int C, int d) const { return ((int64_t)C * (BW + 1) + d) * TILE; }
    __host__ __device__ int n_tiles() const { return nb * (BW + 1); }
};

static TileGeom make_tile_geom(int m1, int m2, int K) {
    TileGeom g;
    g.m1 = m1; g.m2 = m2; g.K = K;
    g.M = m1 * m2;
    g.nb = (g.M + NB - 1) / NB;
    g.w = K * m2 + K;
    g.BW = std::min((g.w + NB - 1) / NB, g.nb - 1);
    return g;
}

// Layout of the factor buffer (`band` of the C ABI), in doubles:
//   [ tiles n_tiles*TILE | Linv nb*TILE | colstat nb*kColStat | flags (ints) ]
// colstat[C] = { 2 sum log L_cc, ||y_C||^2, then %globaltimer stamps (ns) of the diagonal task: begin, operands
// landed, POTRF done, published; and of the first sub-diagonal task: inverse seen, tile published }
struct FactorLayout {
    int64_t tiles, linv, colstat, flags, total;
    int64_t n_flag_ints;
};
static FactorLayout factor_layout(const TileGeom& g) {
    FactorLayout L;
    L.tiles = 0;
    L.linv = (int64_t)g.n_tiles() * TILE;
    L.colstat = L.linv + (int64_t)g.nb * TILE;
    L.flags = L.colstat + (int64_t)g.nb * kColStat;
    L.n_flag_ints = (int64_t)g.n_tiles() + 8 + 2 * (int64_t)g.nb;   // tile flags, abort, first bad pivot, y flags, rhs counters
    L.total = L.flags + (L.n_flag_ints + 1) / 2 + 2;
    return L;
}
// Layout of the selected-inverse buffers: sig = [ lower tiles | upper tiles ], work = [ xacc nb*NB | flags ]
struct SelLayout {
    int64_t sig_lower, sig_upper, sig_total;
    int64_t xacc, flags, work_total, n_flag_ints;
};
static SelLayout sel_layout(const TileGeom& g) {
    SelLayout L;
    L.sig_lower = 0;
    L.sig_upper = (int64_t)g.n_tiles() * TILE;
    L.sig_total = 2 * L.sig_upper;
    L.xacc = 0;
    L.flags = (int64_t)g.nb * NB;
    L.n_flag_ints = (int64_t)g.n_tiles() + 3 * (int64_t)g.nb + 8;   // tile flags, per-column counters, abort, x flags, x counters
    L.work_total = L.flags + (L.n_flag_ints + 1) / 2 + 2;
    return L;
}

// ------------------------------------------------------------------------------------------------------------------
// assembly of P into tiles
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) td_assemble_kernel(TileGeom g, const double* __restrict__ K1,
                                                          const double* __restrict__ K2,
                                                          const double* __restrict__ Gs, double inv_s2,
                                                          double* __restrict__ tiles) {
    const int NS = 2 * g.K + 1;
    const int n_e = (g.K + 1) * NS;
    const int64_t Mpad = (int64_t)g.nb * NB;
    const int64_t total = Mpad * n_e;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t j = t / n_e;
        const int e = (int)(t % n_e);
        const int d1 = e / NS, d2 = e % NS - g.K;
        const int Cb = (int)(j / NB), c = (int)(j % NB);
        if (j >= g.M) {                                     // padding columns: unit diagonal
            if (d1 == 0 && d2 == 0) tiles[g.tile(Cb, 0) + c * NB + c] = 1.0;
            continue;
        }
        if (d1 == 0 && d2 < 0) continue;
        const int j1 = (int)(j / g.m2), j2 = (int)(j % g.m2);
        const int i1 = j1 + d1, i2 = j2 + d2;
        if (i1 >= g.m1 || i2 < 0 || i2 >= g.m2) continue;
        const int a2 = d2 < 0 ? -d2 : d2, c2 = d2 < 0 ? i2 : j2;
        const double kv = K1[(int64_t)d1 * g.m1 + j1] * K2[(int64_t)a2 * g.m2 + c2];
        const double v = fma(inv_s2, Gs[(int64_t)e * g.M + j], kv);
        const int64_t i = j + (int64_t)d1 * g.m2 + d2;
        const int Rb = (int)(i / NB), r = (int)(i % NB);
        tiles[g.tile(Cb, Rb - Cb) + c * NB + r] = v;
        if (Rb == Cb && r != c) tiles[g.tile(Cb, 0) + r * NB + c] = v;     // diagonal tiles are kept full symmetric
    }
}

// ------------------------------------------------------------------------------------------------------------------
// factorisation
// ------------------------------------------------------------------------------------------------------------------
struct FactorArgs {
    TileGeom g;
    double* tiles;      // in: P, out: L
    double* linv;       // nb tiles: L(C,C)^-1 (lower)
    double* rhs;        // in: b (zero padded to nb*NB), out: y = L^-1 b
    double* colstat;    // [nb][2]: 2 sum log L_cc, ||y_C||^2 ; slot [0][..] of the info array below
    int* ready;         // [n_tiles] + abort at [n_tiles]
    double* scal;       // [3]: log|P|, ||y||^2, info  (info written here; sums by td_stats_kernel)
};

__global__ void __launch_bounds__(kTdThreads, 1) td_factor_kernel(FactorArgs a) {
    extern __shared__ __align__(128) unsigned char td_smem[];
    const StageBufs sA{reinterpret_cast<double*>(td_smem)}, sB{reinterpret_cast<double*>(td_smem) + TILE};
    double* const pA = reinterpret_cast<double*>(td_smem) + 4 * TILE;      // padded copies of the operands of the current product
    double* const pB = pA + PTILE;
    __shared__ __align__(8) uint64_t full[2];
    __shared__ double s_vec[NB];
    const TileGeom g = a.g;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tm = (tid & 15) * 4, tn = (tid >> 4) * 4;
    int* abort_flag = a.ready + g.n_tiles();
    // the right-hand side y = L^-1 b rides along as a chain of its own, off the critical path of the tiles:
    // yflag[C] = y_C is final;  rhs_cnt[R] = how many tiles of block row R have subtracted L(R,J) y_J from b_R
    int* yflag = a.ready + g.n_tiles() + 8;
    int* rhs_cnt = yflag + g.nb;
    if (tid == 0) { mbar_init(&full[0], 1); mbar_init(&full[1], 1); }
    fence_proxy_async();
    __syncthreads();
    Phases ph;
    const int n_tasks = g.n_tiles();

    for (int t = blockIdx.x; t < n_tasks; t += gridDim.x) {
        const int C = t / (g.BW + 1), d = t % (g.BW + 1), R = C + d;
        if (R >= g.nb) continue;
        double* my_tile = a.tiles + g.tile(C, d);
        double acc[4][4];
        double* stat = a.colstat + (int64_t)C * kColStat;
        if (tid == 0 && d == 0) stat[2] = global_ns();
        regs_from_tile(acc, my_tile, tm, tn);
        const int J0 = max(0, R - g.BW), nJ = C - J0;

        auto issue = [&](int J, int s) {             // thread 0: wait for the operand tiles, then fetch them by TMA
            wait_flag(a.ready + (int64_t)J * (g.BW + 1) + (R - J), 1, abort_flag);
            if (d != 0) wait_flag(a.ready + (int64_t)J * (g.BW + 1) + (C - J), 1, abort_flag);
            fence_proxy_async();
            mbar_expect_tx(&full[s], d != 0 ? 2 * TILE_BYTES : TILE_BYTES);
            tma_load_tile_(sA[s], a.tiles + g.tile(J, R - J), &full[s]);
            if (d != 0) tma_load_tile_(sB[s], a.tiles + g.tile(J, C - J), &full[s]);
        };
        if (nJ > 0) {
            double cf[8][2] = {};                    // sum_J L(R,J) L(C,J)^T as tensor-core fragments
            if (tid == 0) issue(J0, 0);
            for (int q = 0; q < nJ; ++q) {
                const int s = q & 1;
                if (q + 1 < nJ && tid == 0) issue(J0 + q + 1, s ^ 1);
                mbar_wait(&full[s], ph.get(s));
                ph.flip(s);
                repack_padded(pA, sA[s], tid);
                if (d != 0) repack_padded(pB, sB[s], tid);
                __syncthreads();
                dmma_tile(cf, pA, d != 0 ? pB : pA, warp, lane);
                __syncthreads();
            }
            frags_subtract(acc, cf, sA[0], warp, lane, tm, tn);
        }

        if (d == 0) {
            // ---- diagonal tile: POTRF + inverse in registers, forward substitution of the right-hand side ---------
            double V[4][4];
            double* s11 = sA[0];                     // [16] l + [4] 1/l_cc (+ padding)
            double* spanel = sA[0] + 32;             // [4][64] panel, transposed
            double* swrow = sA[0] + 32 + 4 * NB;     // [4][64]
            double* part = sA[0] + 32 + 8 * NB;      // [16][64]
            __shared__ int s_bad;
            if (tid == 0) { s_bad = -1; stat[3] = global_ns(); }
            __syncthreads();
            potrf_regs(acc, V, tm, tn, s11, spanel, swrow, &s_bad, stat + 8);
            __syncthreads();
            const int first_bad = s_bad;
            if (tid == 0) stat[4] = global_ns();
            // publish L^-1 first (it is what the tiles below wait for), then L (zero above the diagonal)
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (tm + i < tn + j) { acc[i][j] = 0.0; V[i][j] = 0.0; }
                }
            regs_to_tile(V, a.linv + (int64_t)C * TILE, tm, tn);
            __threadfence();
            __syncthreads();
            if (tid == 0) { st_release(a.ready + (int64_t)C * (g.BW + 1), 1); stat[5] = global_ns(); }
            regs_to_tile(acc, my_tile, tm, tn);
            // y_C = L^-1 b_C once every tile of block row C has subtracted its share from b_C
            if (tid == 0) wait_flag(rhs_cnt + C, min(g.BW, C), abort_flag);
            __syncthreads();
            {
                double bv[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) bv[j] = __ldcg(a.rhs + (int64_t)C * NB + tn + j);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    double s = 0.0;
#pragma unroll
                    for (int j = 0; j < 4; ++j) s = fma(V[i][j], bv[j], s);
                    part[(tn >> 2) * NB + tm + i] = s;
                }
            }
            __syncthreads();
            double yv = 0.0, ld = 0.0;
            if (tid < NB) {
                yv = reduce16(part, tid);
                a.rhs[(int64_t)C * NB + tid] = yv;
            }
            __threadfence();
            __syncthreads();
            if (tid == 0) st_release(yflag + C, 1);
            // off the critical path: this block column's share of log|P| and ||y||^2
            if (tm == tn) {
#pragma unroll
                for (int i = 0; i < 4; ++i) ld += log(acc[i][i]);
            }
            double q = yv * yv;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                ld += __shfl_xor_sync(0xffffffffu, ld, o);
                q += __shfl_xor_sync(0xffffffffu, q, o);
            }
            __shared__ double s_ld[kTdThreads / 32], s_q[kTdThreads / 32];
            if ((tid & 31) == 0) { s_ld[tid >> 5] = ld; s_q[tid >> 5] = q; }
            __syncthreads();
            if (tid == 0) {
                double L = 0.0, Q = 0.0;
                for (int wv = 0; wv < kTdThreads / 32; ++wv) { L += s_ld[wv]; Q += s_q[wv]; }
                stat[0] = 2.0 * L;
                stat[1] = Q;
                if (first_bad >= 0) atomicMin(a.ready + g.n_tiles() + 1, C * NB + first_bad + 1);
            }
            __syncthreads();
        } else {
            // ---- off-diagonal tile: L(R,C) = A L(C,C)^-T, then b_R -= L(R,C) y_C ----------------------------------------
            if (tid == 0) {
                wait_flag(a.ready + (int64_t)C * (g.BW + 1), 1, abort_flag);
                if (d == 1) stat[6] = global_ns();
                fence_proxy_async();
                mbar_expect_tx(&full[0], TILE_BYTES);
                tma_load_tile_(sB[0], a.linv + (int64_t)C * TILE, &full[0]);
            }
            regs_to_tile_ld<LDT>(acc, pA, tm, tn);   // A(m, k) at [k*LDT + m]
            __syncthreads();
            mbar_wait(&full[0], ph.get(0));
            ph.flip(0);
            repack_padded(pB, sB[0], tid);
            __syncthreads();
            double L[4][4] = {};
            {
                // L[m][n] = sum_k A[m][k] Linv[n][k] on the tensor cores (this product is on the chain of diagonal tiles)
                double cf[8][2] = {};
                dmma_tile(cf, pA, pB, warp, lane);
                frags_subtract(L, cf, sA[1], warp, lane, tm, tn);  // (stage 1 is idle here)
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) L[i][j] = -L[i][j];
            }
            regs_to_tile(L, my_tile, tm, tn);
            __threadfence();
            __syncthreads();
            if (tid == 0) { st_release(a.ready + (int64_t)C * (g.BW + 1) + d, 1); if (d == 1) stat[7] = global_ns(); }
            // off the critical path: b_R -= L(R,C) y_C as soon as y_C exists
            if (tid == 0) wait_flag(yflag + C, 1, abort_flag);
            __syncthreads();
            if (tid < NB) s_vec[tid] = __ldcg(a.rhs + (int64_t)C * NB + tid);
            __syncthreads();
            double* part = sA[0];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                double s = 0.0;
#pragma unroll
                for (int j = 0; j < 4; ++j) s = fma(L[i][j], s_vec[tn + j], s);
                part[(tn >> 2) * NB + tm + i] = s;
            }
            __syncthreads();
            if (tid < NB) atomicAdd(a.rhs + (int64_t)R * NB + tid, -reduce16(part, tid));
            __threadfence();
            __syncthreads();
            if (tid == 0) red_release_add(rhs_cnt + R, 1);
        }
    }
}

// log|P|, ||y||^2 and the info slot from the per-column statistics (deterministic order)
__global__ void td_stats_kernel(TileGeom g, const double* __restrict__ colstat, const int* __restrict__ ready,
                                double* __restrict__ scal) {
    __shared__ double s0[256], s1[256];
    double a0 = 0.0, a1 = 0.0;
    for (int c = threadIdx.x; c < g.nb; c += blockDim.x) { a0 += colstat[kColStat * c]; a1 += colstat[kColStat * c + 1]; }
    s0[threadIdx.x] = a0; s1[threadIdx.x] = a1;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) { s0[threadIdx.x] += s0[threadIdx.x + o]; s1[threadIdx.x] += s1[threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        scal[0] = s0[0];
        scal[1] = s1[0];
        const int aborted = ready[g.n_tiles()], bad = ready[g.n_tiles() + 1];
        scal[2] = aborted ? -1.0 : (bad != kNoBadPivot ? (double)bad : 0.0);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// selected inverse
// ------------------------------------------------------------------------------------------------------------------
// Pre-pass, one CTA per tile, fully parallel: off-diagonal tiles become Y^T (Y = L(R,C) L(C,C)^-1, stored transposed
// so that it is a plain operand later), diagonal tiles seed Sigma(C,C) = L(C,C)^-T L(C,C)^-1.
__global__ void __launch_bounds__(kTdThreads) td_ypass_kernel(TileGeom g, double* __restrict__ tiles,
                                                              const double* __restrict__ linv,
                                                              double* __restrict__ sig_lower) {
    constexpr int LDP = NB + 1;
    extern __shared__ __align__(16) unsigned char yp_smem[];
    double* sLT = reinterpret_cast<double*>(yp_smem);        // Linv transposed, padded: Linv[k][c] at [k*65 + c]
    double* sL = sLT + NB * LDP;                             // L tile, column-major
    const int C = blockIdx.x / (g.BW + 1), d = blockIdx.x % (g.BW + 1), R = C + d;
    if (R >= g.nb) return;
    const int tid = threadIdx.x, tm = (tid & 15) * 4, tn = (tid >> 4) * 4;
    const double* Li = linv + (int64_t)C * TILE;
    for (int e = tid; e < TILE; e += kTdThreads) sLT[(e % NB) * LDP + e / NB] = Li[e];     // Li[e] = Linv[r=e%64][c=e/64]
    double* T = tiles + g.tile(C, d);
    if (d != 0)
        for (int e = tid; e < TILE; e += kTdThreads) sL[e] = T[e];
    __syncthreads();
    double acc[4][4] = {};
    if (d == 0) {
        // S0[m][n] = sum_k Linv[k][m] Linv[k][n]
        tile_mma<LDP, LDP, false>(acc, sLT, sLT, tm, tn);
        regs_to_tile(acc, sig_lower + g.tile(C, 0), tm, tn);
    } else {
        // Y[m][n] = sum_k L[m][k] Linv[k][n]
        tile_mma<NB, LDP, false>(acc, sL, sLT, tm, tn);
        regs_to_tile_t(acc, T, tm, tn);              // in place: every read of T happened before the barrier above
    }
}

struct SelArgs {
    TileGeom g;
    const double* tiles;    // Y^T tiles (off-diagonal) from the pre-pass
    const double* linv;
    double* sig_lower;      // Sigma(C+d, C) tiles
    double* sig_upper;      // Sigma(C, C+d) tiles (transposes), d >= 1
    double* x;              // in: y = L^-1 b, out: x = P^-1 b
    double* xacc;           // [nb*NB] zeroed: -sum_K Y(K,C)^T x_K
    double* colstat;        // per-block-column record in the factor buffer (slots 12..15: %globaltimer stamps of the d = 1 tile)
    int* sready;            // [n_tiles] tile flags, [nb] column counters, abort
};

__global__ void __launch_bounds__(kTdThreads, 1) td_selinv_kernel(SelArgs a) {
    extern __shared__ __align__(128) unsigned char td_smem[];
    const StageBufs sA{reinterpret_cast<double*>(td_smem)}, sB{reinterpret_cast<double*>(td_smem) + TILE};
    double* const pA = reinterpret_cast<double*>(td_smem) + 4 * TILE;      // padded copies of the operands of the current product
    double* const pB = pA + PTILE;
    __shared__ __align__(8) uint64_t full[2];
    __shared__ double s_vec[NB];
    const TileGeom g = a.g;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tm = (tid & 15) * 4, tn = (tid >> 4) * 4;
    int* cnt = a.sready + g.n_tiles();            // cnt[C]: off-diagonal tiles of column C that have added their share to Sigma(C,C)
    int* abort_flag = cnt + g.nb;
    // the back substitution x = P^-1 b is a chain of its own, off the critical path of the tiles:
    // xflag[C] = x_C is final;  xcnt[C] = off-diagonal tiles of column C that have added -Y(K,C)^T x_K
    int* xflag = abort_flag + 8;
    int* xcnt = xflag + g.nb;
    if (tid == 0) { mbar_init(&full[0], 1); mbar_init(&full[1], 1); }
    fence_proxy_async();
    __syncthreads();
    Phases ph;
    const int n_tasks = g.n_tiles();

    for (int t = blockIdx.x; t < n_tasks; t += gridDim.x) {
        // order: block columns descending; inside a column the off-diagonal tiles first (far to near), the diagonal last
        const int C = g.nb - 1 - t / (g.BW + 1);
        const int d = g.BW - t % (g.BW + 1);
        const int R = C + d;
        if (R >= g.nb) continue;
        const int Kmax = min(g.nb - 1, C + g.BW);

        if (d != 0) {
            const int nK = Kmax - C;
            double* sstat = a.colstat + (int64_t)C * kColStat;
            auto issue = [&](int K, int s) {         // A = Sigma(R, K), B = Y(K, C)^T
                const double* src;
                const int* flag;
                int want = 1;
                if (K == R) { src = a.sig_lower + g.tile(R, 0); flag = cnt + R; want = min(g.BW, g.nb - 1 - R); }   // Sigma(R,R): all shares in
                else if (K < R) { src = a.sig_lower + g.tile(K, R - K); flag = a.sready + (int64_t)K * (g.BW + 1) + (R - K); }
                else { src = a.sig_upper + g.tile(R, K - R); flag = a.sready + (int64_t)R * (g.BW + 1) + (K - R); }
                // the Y^T operand is there since the pre-pass: it is requested before the wait, only Sigma(R,K) after it
                mbar_expect_tx(&full[s], 2 * TILE_BYTES);
                tma_load_tile_(sB[s], a.tiles + g.tile(C, K - C), &full[s]);
                if (d == 1 && K == R) sstat[16] = global_ns();              // starts waiting for Sigma(R,R)
                wait_flag(flag, want, abort_flag);
                if (d == 1 && K == R) sstat[17] = global_ns();              // ... complete
                fence_proxy_async();
                tma_load_tile_(sA[s], src, &full[s]);
                if (d == 1 && K == R) sstat[18] = global_ns();              // copy issued
            };
            double acc[4][4] = {};
            double cf[8][2] = {};                    // sum_K Sigma(R,K) Y(K,C) as tensor-core fragments
            if (tid == 0) issue(Kmax, 0);
            for (int q = 0; q < nK; ++q) {
                const int s = q & 1;
                if (tid == 0) {
                    if (q + 1 < nK) {
                        issue(Kmax - q - 1, s ^ 1);
                    } else {
                        // last product: the idle stage already fetches this tile's own Y^T for the diagonal contribution below
                        mbar_expect_tx(&full[s ^ 1], TILE_BYTES);
                        tma_load_tile_(sB[s ^ 1], a.tiles + g.tile(C, d), &full[s ^ 1]);
                    }
                }
                mbar_wait(&full[s], ph.get(s));
                ph.flip(s);
                if (tid == 0 && d == 1 && q + 1 == nK) sstat[12] = global_ns();     // operands of the last product (Sigma(R,R)) landed
                if (Kmax - q == R) repack_padded_sym(pA, sA[s], tid);      // Sigma(R,R): enforce symmetry (see repack_padded_sym)
                else repack_padded(pA, sA[s], tid);
                repack_padded(pB, sB[s], tid);
                __syncthreads();
                dmma_tile(cf, pA, pB, warp, lane);
                __syncthreads();
            }
            const int so = nK & 1;                                          // the stage holding the own tile
            frags_subtract(acc, cf, sA[so ^ 1], warp, lane, tm, tn);       // acc = -sum_K Sigma(R,K) Y(K,C)
            if (tid == 0 && d == 1) sstat[13] = global_ns();
            // Sigma(R, C) = acc: publish both orientations
            regs_to_tile(acc, a.sig_lower + g.tile(C, d), tm, tn);
            // the transpose goes through shared memory (it is needed there anyway, as an operand of the diagonal contribution
            // below) and leaves as whole 512-byte columns; 16-byte stores straight from the registers made the publish 3.8 us
            regs_to_tile_t_ld<LDT>(acc, pA, tm, tn);         // T[m][a] at [m*LDT + a]  ==  A'(a, k=m) at [k*LDT + a]
            __syncthreads();
            {
                double* up = a.sig_upper + g.tile(C, d);
#pragma unroll
                for (int idx = tid; idx < TILE / 2; idx += kTdThreads) {
                    const int c = idx >> 5, r = (idx & 31) * 2;
                    *reinterpret_cast<double2*>(up + c * NB + r) = *reinterpret_cast<const double2*>(pA + c * LDT + r);
                }
            }
            __threadfence();
            __syncthreads();
            if (tid == 0) { st_release(a.sready + (int64_t)C * (g.BW + 1) + d, 1); if (d == 1) sstat[14] = global_ns(); }
            mbar_wait(&full[so], ph.get(so));
            ph.flip(so);
            repack_padded(pB, sB[so], tid);
            __syncthreads();
            {
                // D[a][b] = sum_m T[m][a] Y[m][b] on the tensor cores (this product is on the chain of diagonal tiles); the
                // fragments go straight to the diagonal tile as REDs
                double D[8][2] = {};
                dmma_tile(D, pA, pB, warp, lane);
                double* Sd = a.sig_lower + g.tile(C, 0);
                const int row = warp * 8 + (lane >> 2), col = (lane & 3) * 2;
#pragma unroll
                for (int cb = 0; cb < 8; ++cb) {
                    atomicAdd(Sd + (cb * 8 + col) * NB + row, -D[cb][0]);
                    atomicAdd(Sd + (cb * 8 + col + 1) * NB + row, -D[cb][1]);
                }
            }
            __threadfence();
            __syncthreads();
            if (tid == 0) { red_release_add(cnt + C, 1); if (d == 1) sstat[15] = global_ns(); }
            // off the critical path: xacc_C[b] -= sum_m Y[m][b] x_R[m] as soon as x_R exists;  Y[m][b] at sB[so][m*64 + b]
            if (tid == 0) wait_flag(xflag + R, 1, abort_flag);
            __syncthreads();
            if (tid < NB) s_vec[tid] = __ldcg(a.x + (int64_t)R * NB + tid);
            __syncthreads();
            if (tid < NB) {
                double s = 0.0;
#pragma unroll 8
                for (int m = 0; m < NB; ++m) s = fma(sB[so][m * NB + tid], s_vec[m], s);
                atomicAdd(a.xacc + (int64_t)C * NB + tid, -s);
            }
            __threadfence();
            __syncthreads();
            if (tid == 0) red_release_add(xcnt + C, 1);
        } else {
            // diagonal task: only the back substitution is left to do (Sigma(C,C) is complete when cnt[C] is, which is
            // what its readers wait for)
            if (tid == 0) wait_flag(xcnt + C, Kmax - C, abort_flag);
            __syncthreads();
            // x_C = L(C,C)^-T y_C + xacc_C
            double V[4][4];
            regs_from_tile(V, a.linv + (int64_t)C * TILE, tm, tn);
            double* part = sA[0];
            if (tid < NB) s_vec[tid] = a.x[(int64_t)C * NB + tid];
            __syncthreads();
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                double s = 0.0;
#pragma unroll
                for (int i = 0; i < 4; ++i) s = fma(V[i][j], s_vec[tm + i], s);
                part[(tm >> 2) * NB + tn + j] = s;
            }
            __syncthreads();
            if (tid < NB) {
                const double xa = __ldcg(a.xacc + (int64_t)C * NB + tid);
                a.x[(int64_t)C * NB + tid] = reduce16(part, tid) + xa;
            }
            __threadfence();
            __syncthreads();
            if (tid == 0) st_release(xflag + C, 1);
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// stencil extraction and the scalar contractions needed by the gradients
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) td_extract_stencil_kernel(TileGeom g, const double* __restrict__ sig_lower,
                                                                 const int* __restrict__ abort_flag,
                                                                 double* __restrict__ out) {
    const int NS = 2 * g.K + 1, n_e = (g.K + 1) * NS;
    const int64_t total = (int64_t)g.M * n_e;
    const bool aborted = *abort_flag != 0;       // the persistent kernel gave up waiting: poison the result
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int e = (int)(t / g.M);
        const int64_t j = t % g.M;
        const int d1 = e / NS, d2 = e % NS - g.K;
        const int j1 = (int)(j / g.m2), j2 = (int)(j % g.m2);
        const int i1 = j1 + d1, i2 = j2 + d2;
        double v = 0.0;
        if (!(d1 == 0 && d2 < 0) && i1 < g.m1 && i2 >= 0 && i2 < g.m2) {
            const int64_t i = j + (int64_t)d1 * g.m2 + d2;
            const int Cb = (int)(j / NB), c = (int)(j % NB), Rb = (int)(i / NB), r = (int)(i % NB);
            v = __ldcg(sig_lower + g.tile(Cb, Rb - Cb) + c * NB + r);
            if (Rb == Cb) v = 0.5 * (v + __ldcg(sig_lower + g.tile(Cb, 0) + r * NB + c));   // diagonal tiles: see repack_padded_sym
        }
        out[t] = aborted ? nan("") : v;
    }
}

// For the stencil operators  Op in { G,  dK1 (x) K2,  K1 (x) dK2,  K1 (x) K2 }  and a symmetric stencil field S:
//   out[o]     = sum_{i,j} S[i,j] Op[i,j]   (full symmetric sum = diagonal once + off-diagonals twice)
//   out[4 + o] = x^T Op x
// plus the Kronecker trace terms  out[8..10] = sum G[(i),(j)] T1[i1,j1] T2[i2,j2] for (T1,T2) in
//   (S1,S2), (dS1,S2), (S1,dS2)   (reference gpr.py:307 trace(cholesky_solve(L_Kuu, KufKfu)) and its derivatives).
// A batch (asvgp_kron_terms_batched): blockIdx.y = b D + d for slot b and output column d; slot b reads SigP + b sig_stride, the
// per-dimension bands + b k1_stride / k2_stride, x + (b D + d) M, and writes out + (b D + d) 11.  Gs is shared.
struct StencilTerms {
    const double *SigP, *Gs, *x;
    const double *K1, *dK1, *K2, *dK2;        // lower bands (K+1) x m
    const double *S1, *dS1, *S2, *dS2;        // lower bands of K1^-1, d(K1^-1), K2^-1, d(K2^-1)
    long long sig_stride, k1_stride, k2_stride;
    int n_cols;
};

__device__ __forceinline__ double band_sym(const double* B, int m, int i, int j) {
    const int d = i - j;
    return d >= 0 ? B[(int64_t)d * m + j] : B[(int64_t)(-d) * m + i];
}

__global__ void __launch_bounds__(256) td_terms_kernel(int m1, int m2, int K, StencilTerms a, double* __restrict__ out) {
    const int NS = 2 * K + 1, n_e = (K + 1) * NS;
    const int64_t M = (int64_t)m1 * m2;
    const int64_t total = M * n_e;
    {
        const int b = blockIdx.y / a.n_cols;
        a.SigP += b * a.sig_stride;
        a.x += blockIdx.y * M;
        a.K1 += b * a.k1_stride; a.dK1 += b * a.k1_stride; a.S1 += b * a.k1_stride; a.dS1 += b * a.k1_stride;
        a.K2 += b * a.k2_stride; a.dK2 += b * a.k2_stride; a.S2 += b * a.k2_stride; a.dS2 += b * a.k2_stride;
        out += blockIdx.y * 11;
    }
    double acc[11];
#pragma unroll
    for (int i = 0; i < 11; ++i) acc[i] = 0.0;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int e = (int)(t / M);
        const int64_t j = t % M;
        const int d1 = e / NS, d2 = e % NS - K;
        if (d1 == 0 && d2 < 0) continue;
        const int j1 = (int)(j / m2), j2 = (int)(j % m2);
        const int i1 = j1 + d1, i2 = j2 + d2;
        if (i1 >= m1 || i2 < 0 || i2 >= m2) continue;
        const int64_t i = (int64_t)i1 * m2 + i2;
        const double wgt = (d1 == 0 && d2 == 0) ? 1.0 : 2.0;
        const double s = a.SigP[t], gv = a.Gs[t];
        const double k1 = a.K1[(int64_t)d1 * m1 + j1], dk1 = a.dK1[(int64_t)d1 * m1 + j1];
        const double k2 = band_sym(a.K2, m2, i2, j2), dk2 = band_sym(a.dK2, m2, i2, j2);
        const double xx = wgt * a.x[i] * a.x[j], ws = wgt * s;
        const double op[4] = {gv, dk1 * k2, k1 * dk2, k1 * k2};
#pragma unroll
        for (int o = 0; o < 4; ++o) { acc[o] = fma(ws, op[o], acc[o]); acc[4 + o] = fma(xx, op[o], acc[4 + o]); }
        const double s1 = a.S1[(int64_t)d1 * m1 + j1], ds1 = a.dS1[(int64_t)d1 * m1 + j1];
        const double s2 = band_sym(a.S2, m2, i2, j2), ds2 = band_sym(a.dS2, m2, i2, j2);
        const double wg = wgt * gv;
        acc[8] = fma(wg, s1 * s2, acc[8]);
        acc[9] = fma(wg, ds1 * s2, acc[9]);
        acc[10] = fma(wg, s1 * ds2, acc[10]);
    }
    __shared__ double s_red[11][8];
#pragma unroll
    for (int i = 0; i < 11; ++i) {
        double v = acc[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0) s_red[i][threadIdx.x >> 5] = v;
    }
    __syncthreads();
    if (threadIdx.x < 11) {
        double v = 0.0;
        for (int wv = 0; wv < 8; ++wv) v += s_red[threadIdx.x][wv];
        atomicAdd(out + threadIdx.x, v);
    }
}


}  // namespace asvgp

using namespace asvgp;

extern "C" int64_t asvgp_kronband_band_doubles(int m1, int m2, int order) {
    if (m1 <= 0 || m2 <= 0 || order < 1 || order > kMaxOrder) return -1;
    return factor_layout(make_tile_geom(m1, m2, order)).total;
}
// Diagnostics: offset (doubles) of the per-block-column statistics inside `band`; 8 doubles per block column, see
// factor_layout.  n_block_columns = ceil(m1*m2 / 64).
extern "C" int64_t asvgp_kronband_colstat_offset(int m1, int m2, int order) {
    if (m1 <= 0 || m2 <= 0 || order < 1 || order > kMaxOrder) return -1;
    return factor_layout(make_tile_geom(m1, m2, order)).colstat;
}
extern "C" int64_t asvgp_kronband_sig_doubles(int m1, int m2, int order) {
    if (m1 <= 0 || m2 <= 0 || order < 1 || order > kMaxOrder) return -1;
    return sel_layout(make_tile_geom(m1, m2, order)).sig_total;
}
extern "C" int64_t asvgp_kronband_work_doubles(int m1, int m2, int order) {
    if (m1 <= 0 || m2 <= 0 || order < 1 || order > kMaxOrder) return -1;
    return sel_layout(make_tile_geom(m1, m2, order)).work_total;
}
extern "C" int64_t asvgp_kronband_rhs_doubles(int m1, int m2, int order) {
    if (m1 <= 0 || m2 <= 0 || order < 1 || order > kMaxOrder) return -1;
    return (int64_t)make_tile_geom(m1, m2, order).nb * NB;
}

// Assembles P into `band` (asvgp_kron_band_doubles doubles) and factorises it in place.
// rhs_io[asvgp_kron_rhs_doubles]: in = Kuf_y (zero padded), out = y = L^-1 Kuf_y.  scal[3] = log|P|, ||y||^2, info.
extern "C" int asvgp_kronband_factor(const double* K1, const double* K2, const double* Gs, int m1, int m2, int order,
                                 double sigma2, double* band, double* rhs_io, double* scal, void* stream) {
    ASVGP_REQUIRE(m1 > 0 && m2 > 0 && order >= 1 && order <= kMaxOrder, "kronband_factor: m=%d,%d order=%d", m1, m2, order);
    ASVGP_REQUIRE(sigma2 > 0.0, "kronband_factor: sigma2=%g", sigma2);
    const TileGeom g = make_tile_geom(m1, m2, order);
    const FactorLayout lay = factor_layout(g);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int* flags = reinterpret_cast<int*>(band + lay.flags);
    ASVGP_CUDA_OK(cudaMemsetAsync(band, 0, (size_t)lay.linv * sizeof(double), st));                       // tiles
    ASVGP_CUDA_OK(cudaMemsetAsync(flags, 0, (size_t)lay.n_flag_ints * sizeof(int), st));
    ASVGP_CUDA_OK(cudaMemsetAsync(flags + g.n_tiles() + 1, 0x7f, sizeof(int), st));                       // first bad pivot = "none"
    const int64_t total = (int64_t)g.nb * NB * (order + 1) * (2 * order + 1);
    td_assemble_kernel<<<(int)std::min<int64_t>((total + 255) / 256, 148 * 16), 256, 0, st>>>(g, K1, K2, Gs, 1.0 / sigma2, band); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    FactorArgs a{g, band, band + lay.linv, rhs_io, band + lay.colstat, flags, scal};
    int grid = 0;
    if (int rc = persistent_grid(td_factor_kernel, kTdSmem, g.n_tiles(), &grid)) return rc;
    void* params[] = {&a};
    ASVGP_CUDA_OK(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(td_factor_kernel), dim3(grid), dim3(kTdThreads),
                                              params, kTdSmem, st));
    ASVGP_LAUNCHED();
    td_stats_kernel<<<1, 256, 0, st>>>(g, band + lay.colstat, flags, scal); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

// From the factor (overwritten: its off-diagonal tiles become Y^T): sigma_stencil[(order+1)(2 order+1) x M] = entries of
// P^-1 on the stencil, x_io: in y = L^-1 b, out x = P^-1 b.  sig_band: asvgp_kron_sig_doubles doubles of scratch;
// work: asvgp_kron_work_doubles doubles.  If the persistent kernel gives up waiting (abort flag), sigma_stencil is
// filled with NaN.
extern "C" int asvgp_kronband_selinv(double* band, int m1, int m2, int order, double* sig_band, double* x_io,
                                 double* sigma_stencil, double* work, void* stream) {
    ASVGP_REQUIRE(m1 > 0 && m2 > 0 && order >= 1 && order <= kMaxOrder, "kronband_selinv: m=%d,%d order=%d", m1, m2, order);
    const TileGeom g = make_tile_geom(m1, m2, order);
    const FactorLayout fl = factor_layout(g);
    const SelLayout sl = sel_layout(g);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int* flags = reinterpret_cast<int*>(work + sl.flags);
    ASVGP_CUDA_OK(cudaMemsetAsync(work, 0, (size_t)sl.work_total * sizeof(double), st));                  // xacc + flags
    const size_t yp_smem = (size_t)(NB * (NB + 1) + TILE) * sizeof(double);
    ASVGP_CUDA_OK(cudaFuncSetAttribute(td_ypass_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)yp_smem));
    td_ypass_kernel<<<g.n_tiles(), kTdThreads, yp_smem, st>>>(g, band, band + fl.linv, sig_band + sl.sig_lower); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    SelArgs a{g, band, band + fl.linv, sig_band + sl.sig_lower, sig_band + sl.sig_upper, x_io, work + sl.xacc, band + fl.colstat, flags};
    int grid = 0;
    if (int rc = persistent_grid(td_selinv_kernel, kTdSmem, g.n_tiles(), &grid)) return rc;
    void* params[] = {&a};
    ASVGP_CUDA_OK(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(td_selinv_kernel), dim3(grid), dim3(kTdThreads),
                                              params, kTdSmem, st));
    ASVGP_LAUNCHED();
    const int64_t total = (int64_t)g.M * (order + 1) * (2 * order + 1);
    td_extract_stencil_kernel<<<(int)std::min<int64_t>((total + 255) / 256, 148 * 16), 256, 0, st>>>(
        g, sig_band + sl.sig_lower, flags + g.n_tiles() + g.nb, sigma_stencil); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

// out[11] (device, zeroed here): see td_terms_kernel.
extern "C" int asvgp_kron_terms(const double* SigP, const double* Gs, const double* x, const double* K1,
                                const double* dK1, const double* K2, const double* dK2, const double* S1,
                                const double* dS1, const double* S2, const double* dS2, int m1, int m2, int order,
                                double* out, void* stream) {
    ASVGP_REQUIRE(m1 > 0 && m2 > 0 && order >= 1 && order <= kMaxOrder, "kron_terms: m=%d,%d order=%d", m1, m2, order);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ASVGP_CUDA_OK(cudaMemsetAsync(out, 0, 11 * sizeof(double), st));
    StencilTerms a{SigP, Gs, x, K1, dK1, K2, dK2, S1, dS1, S2, dS2, 0, 0, 0, 1};
    const int64_t total = (int64_t)m1 * m2 * (order + 1) * (2 * order + 1);
    td_terms_kernel<<<(int)std::min<int64_t>((total + 255) / 256, 148 * 4), 256, 0, st>>>(m1, m2, order, a, out); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

// B settings x D output columns in one launch: SigP[B][(order+1)(2 order+1)][M], x[B][D][M], per-dimension bands [B][order+1][m_i],
// Gs shared; out[B][D][11] (device, zeroed here), entry (b, d) as asvgp_kron_terms on slot b's operands and column d.
extern "C" int asvgp_kron_terms_batched(const double* SigP, const double* Gs, const double* x, const double* K1,
                                        const double* dK1, const double* K2, const double* dK2, const double* S1,
                                        const double* dS1, const double* S2, const double* dS2, int m1, int m2, int order,
                                        int B, int D, double* out, void* stream) {
    ASVGP_REQUIRE(m1 > 0 && m2 > 0 && order >= 1 && order <= kMaxOrder, "kron_terms_batched: m=%d,%d order=%d", m1, m2, order);
    ASVGP_REQUIRE(B >= 1 && B <= ASVGP_MAX_BATCH, "kron_terms_batched: B=%d not in 1..%d", B, ASVGP_MAX_BATCH);
    ASVGP_REQUIRE(D >= 1 && D <= ASVGP_MAX_RHS, "kron_terms_batched: D=%d not in 1..%d", D, ASVGP_MAX_RHS);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ASVGP_CUDA_OK(cudaMemsetAsync(out, 0, (size_t)B * D * 11 * sizeof(double), st));
    const int n_e = (order + 1) * (2 * order + 1);
    StencilTerms a{SigP, Gs, x, K1, dK1, K2, dK2, S1, dS1, S2, dS2, (long long)n_e * m1 * m2, (long long)(order + 1) * m1,
                   (long long)(order + 1) * m2, D};
    const int64_t total = (int64_t)m1 * m2 * n_e;
    const int per = (int)std::max<int64_t>(1, std::min<int64_t>((total + 255) / 256, (148 * 4 + B * D - 1) / (B * D)));
    td_terms_kernel<<<dim3(per, B * D), 256, 0, st>>>(m1, m2, order, a, out); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}
