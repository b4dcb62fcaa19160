// Latency-bound banded kernels of the 1-D model: Kuu assembly, collapsed ELBO + hyper-parameter gradients,
// posterior weights for the predictor.
//
//   asvgp_kuu_assemble   <- SplineFeatures1D.make_Kuu                    (reference asvgp/inducing_features.py:12-44)
//   asvgp_elbo_grad_1d   <- GPR_1d.elbo + its TF-autodiff gradient       (reference asvgp/gpr.py:49-89, example.py:31-32)
//   asvgp_posterior_1d   <- the factorisations/solves of GPR_1d.predict_f (reference asvgp/gpr.py:96-108)
//   asvgp_kuu_assemble_batched, asvgp_elbo_grad_1d_batched: the first two for B hyper-parameter settings at once
//
// Design (DESIGN.md §4.2).  The work is O(M k^2) flops — nothing — but a length-M dependency chain of
// sqrt/div/FMA.  Each "chain" (one SPD banded matrix) runs in ONE CTA through the partitioned engine of
// band_engine.cuh: P lanes eliminate P chunks in lock-step, lane 0 eliminates the (P-1)k separator system, the lanes
// sweep back.  Independent chains run in different CTAs of the same launch:
//   ELBO+grad : [Kuu, d/dl] with Takahashi + trace,  [P, d/dl] forward only,  [P, d/dsigma2] forward only
//   posterior : [Kuu] Takahashi,  [P] solve + Takahashi
// Derivatives ride along as Dual<1> tangents; the variance derivative follows analytically from the sigma2 one
// because Kuu is proportional to 1/variance (see elbo_finalize_kernel).
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>

#include <algorithm>

#include "band_engine.cuh"
#include "../../include/asvgp_b200.h"

namespace asvgp {

constexpr int kChainThreads = 128;          // >= max chunk count P

// programmatic dependent launch (see launch_dependent): no-ops when the kernel was launched the ordinary way
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
constexpr int kMaxTerms = 12;

// ------------------------------------------------------------------------------------------------------------------
// Kuu assembly
// ------------------------------------------------------------------------------------------------------------------
struct KuuTerms {
    int n_terms;
    double coef[kMaxTerms];
    double dcoef[kMaxTerms];
};

// One coefficient set per slot of a batch (asvgp_kuu_assemble_batched): ~12 KB of kernel parameters at ASVGP_MAX_BATCH.
struct KuuTermsBatch {
    int n_terms;
    double coef[ASVGP_MAX_BATCH][kMaxTerms];
    double dcoef[ASVGP_MAX_BATCH][kMaxTerms];
};

__device__ __forceinline__ void kuu_assemble_band(const double* __restrict__ tables, int n_terms, const double* coef,
                                                  const double* dcoef, int64_t band_elems, double* __restrict__ Kuu,
                                                  double* __restrict__ dKuu) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < band_elems;
         i += (int64_t)gridDim.x * blockDim.x) {
        // The reference's own operation order (inducing_features.py:17-44: every term `coefficient * table` rounded, then
        // summed left to right) instead of a fused multiply-add chain: at l / delta ~ 18 the bound moves by a few 1e-10
        // relative per ulp of Kuu (cond(Kuu) ~ 6e4 against 1 / sigma2), so the assembly should round where the
        // reference's does.
        double v = 0.0, dv = 0.0;
        for (int t = 0; t < n_terms; ++t) {
            const double s = __ldg(tables + (int64_t)t * band_elems + i);
            v = __dadd_rn(v, __dmul_rn(coef[t], s));
            dv = __dadd_rn(dv, __dmul_rn(dcoef[t], s));
        }
        Kuu[i] = v;
        if (dKuu != nullptr) dKuu[i] = dv;
    }
}

__global__ void __launch_bounds__(256) kuu_assemble_kernel(const double* __restrict__ tables, const __grid_constant__ KuuTerms terms,
                                                           int64_t band_elems, double* __restrict__ Kuu,
                                                           double* __restrict__ dKuu) {
    kuu_assemble_band(tables, terms.n_terms, terms.coef, terms.dcoef, band_elems, Kuu, dKuu);
}

// slot = blockIdx.y: the band of slot b is Kuu[b] of [B, k+1, M], entry for entry the operations of kuu_assemble_kernel
__global__ void __launch_bounds__(256) kuu_assemble_batched_kernel(const double* __restrict__ tables, const __grid_constant__ KuuTermsBatch terms,
                                                                   int64_t band_elems, double* __restrict__ Kuu,
                                                                   double* __restrict__ dKuu) {
    const int b = blockIdx.y;
    kuu_assemble_band(tables, terms.n_terms, terms.coef[b], terms.dcoef[b], band_elems, Kuu + b * band_elems,
                      dKuu != nullptr ? dKuu + b * band_elems : nullptr);
}

// ------------------------------------------------------------------------------------------------------------------
// matrix / right-hand-side functors fed to the engine
// ------------------------------------------------------------------------------------------------------------------
// All accessors are branch-free (clamped index + select) so that the loads of one window row issue back to back
// and can be hoisted two columns ahead of their use.
template <class T> struct BandMat;      // A = Kuu + beta*G  with tangent  use_dK*dKuu + tb*G
template <> struct BandMat<Dual<1>> {
    const double* Kuu; const double* dKuu; const double* G;
    double beta, tb; int use_dK; int M;
    __device__ __forceinline__ Dual<1> operator()(int d, int j) const {
        const bool ok = (j >= 0) & (j + d < M);
        const size_t i = ok ? (size_t)d * M + j : 0;
        const double kv = __ldg(Kuu + i);
        const double dk = use_dK ? __ldg(dKuu + i) : 0.0;
        const double g = (G != nullptr) ? __ldg(G + i) : 0.0;
        Dual<1> r;
        r.v = ok ? fma(beta, g, kv) : 0.0;
        r.d[0] = ok ? fma(tb, g, dk) : 0.0;
        return r;
    }
};
template <> struct BandMat<double> {
    const double* Kuu; const double* dKuu; const double* G;
    double beta, tb; int use_dK; int M;
    __device__ __forceinline__ double operator()(int d, int j) const {
        const bool ok = (j >= 0) & (j + d < M);
        const size_t i = ok ? (size_t)d * M + j : 0;
        const double kv = __ldg(Kuu + i);
        const double g = (G != nullptr) ? __ldg(G + i) : 0.0;
        return ok ? fma(beta, g, kv) : 0.0;
    }
};
template <class T> struct VecRhs {      // use == 0: zero right-hand side (b must still be a readable pointer)
    const double* b; int M; int use;
    __device__ __forceinline__ T operator()(int j) const {
        const bool ok = (use != 0) & (j >= 0) & (j < M);
        const double v = __ldg(b + (ok ? j : 0));
        return make_scalar<T>(ok ? v : 0.0, 0.0);
    }
};

// ------------------------------------------------------------------------------------------------------------------
// lane-interleaved row tables
// ------------------------------------------------------------------------------------------------------------------
// The P lanes of a chain sweep P different chunks in lock-step, so reading the band directly costs 32 separate sectors
// per load instruction (the sweeps were LSU-bound: per-column time GREW with P).  A fully parallel pre-pass therefore
// tabulates, for every chain, what lane p needs at row rho of its chunk —
//     rows[(rho * (K+1) + bidx) * P + p] = A[g0(p) + rho, g0(p) + rho - K + bidx],     rhs[rho * P + p] = b[g0(p) + rho]
// — and the sweeps read those tables with fully coalesced loads.  Every access A(d, col) of the engine maps to
// rho = col + d - g0, bidx = K - d.
template <class T, int K>
struct RowsMat {
    const T* rows; int g0, P, p, n_rho;
    __device__ __forceinline__ T operator()(int d, int col) const {
        const int rho = col + d - g0;
        const bool ok = (rho >= 0) & (rho < n_rho);
        const T v = rows[ok ? ((size_t)rho * (K + 1) + (K - d)) * P + p : (size_t)p];      // branch-free
        return ok ? v : zero_of<T>();
    }
};
template <class T>
struct RowsRhs {
    const T* r; int g0, P, p, n_rho;
    __device__ __forceinline__ T operator()(int j) const {
        const int rho = j - g0;
        const bool ok = (rho >= 0) & (rho < n_rho);
        const T v = r[ok ? (size_t)rho * P + p : (size_t)p];
        return ok ? v : zero_of<T>();
    }
};
__host__ __device__ inline int chain_n_rho(const ChunkLayout& lay, int K) { return lay.max_size() + K + 4; }
template <class T, int K>
__host__ __device__ inline size_t chain_rows_count(const ChunkLayout& lay) {
    return (size_t)chain_n_rho(lay, K) * (K + 2) * lay.P;            // (K+1) window entries + the right-hand side
}

template <class T> struct ChainSpec { BandMat<T> A; VecRhs<T> rhs; };

// trace(Kuu^-1 G) = sum band(Kuu^-1) .* band(G) (off-diagonals twice, reference gpr.py:60-70) and its d/dl from the stored
// inverse band of the Kuu chain: kTraceBlocks CTAs of 256 threads, every thread a fixed strided share with all its loads in
// flight at once, fixed-order trees; the per-CTA partials are added in CTA order by elbo_finalize_kernel — the same bits on
// every run and every rank, whichever kernel hosts the CTAs (the P chains' chain_rows_kernel or the finalize kernel itself).
constexpr int kTraceBlocks = 64, kTraceThreads = 256, kTraceUnroll = 4;
struct TraceJob {
    const double* kstate;   // nullptr: no trace CTAs in this launch
    const double* G;
    double* tr_part;        // [kTraceBlocks][2]
    int M, K, first_block;
};
__device__ __forceinline__ void trace_partial(const double* __restrict__ kstate, const double* __restrict__ G, int M, int K, int block,
                                              double* __restrict__ tr_part) {
    __shared__ double s_tr[2][kTraceThreads / 32];
    const Dual<1>* kinv = reinterpret_cast<const Dual<1>*>(kstate + 16);
    double tr = 0.0, dtr_dl = 0.0;
    const int band = (K + 1) * M, stride = kTraceThreads * kTraceBlocks;
    for (int i0 = block * kTraceThreads + threadIdx.x; i0 < band; i0 += stride * kTraceUnroll) {
        Dual<1> sv[kTraceUnroll];
        double gv[kTraceUnroll];
#pragma unroll
        for (int u = 0; u < kTraceUnroll; ++u) {
            const int i = i0 + u * stride;
            const int d = i / M, col = i - d * M;
            const bool ok = i < band && col + d < M;
            sv[u] = kinv[ok ? i : 0];
            gv[u] = ok ? (d == 0 ? 1.0 : 2.0) * G[i] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < kTraceUnroll; ++u) {
            if (gv[u] != 0.0) { tr = fma(sv[u].v, gv[u], tr); dtr_dl = fma(sv[u].d[0], gv[u], dtr_dl); }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        tr += __shfl_xor_sync(0xffffffffu, tr, o);
        dtr_dl += __shfl_xor_sync(0xffffffffu, dtr_dl, o);
    }
    if ((threadIdx.x & 31) == 0) { s_tr[0][threadIdx.x >> 5] = tr; s_tr[1][threadIdx.x >> 5] = dtr_dl; }
    __syncthreads();
    if (threadIdx.x == 0) {
        tr = 0.0; dtr_dl = 0.0;
        for (int i = 0; i < kTraceThreads / 32; ++i) { tr += s_tr[0][i]; dtr_dl += s_tr[1][i]; }
        tr_part[2 * block] = tr; tr_part[2 * block + 1] = dtr_dl;
    }
}

// Entry e of one chain's row table (layout above).
template <class T, int K>
__device__ __forceinline__ T chain_rows_entry(const ChunkLayout& lay, const ChainSpec<T>& sp, unsigned e) {
    const unsigned n_rho = chain_n_rho(lay, K), P = lay.P;
    const unsigned q = e / P;
    const int p = (int)(e - q * P);
    const int g0 = P > 1 ? lay.start(p) : 0;
    if (q < n_rho * (K + 1)) {
        const int rho = (int)(q / (K + 1)), bidx = (int)(q - (unsigned)rho * (K + 1));
        const int row = g0 + rho, col = row - K + bidx;
        return sp.A(K - bidx, col);
    }
    const int rho = (int)(q - n_rho * (K + 1));
    return sp.rhs(g0 + rho);
}

template <class T, int K, int NCHAINS>
__global__ void __launch_bounds__(256) chain_rows_kernel(ChunkLayout lay, ChainSpec<T> s0, ChainSpec<T> s1, ChainSpec<T> s2, ChainSpec<T> s3,
                                                         T* __restrict__ out, unsigned* __restrict__ zero_me = nullptr,
                                                         TraceJob trace = TraceJob{nullptr, nullptr, nullptr, 0, 0, 0}) {
    pdl_launch_dependents();
    if (zero_me != nullptr && blockIdx.x == 0 && threadIdx.x == 0) *zero_me = 0u;      // arrival counter of elbo_finalize_kernel
    if (trace.kstate != nullptr && (int)blockIdx.x >= trace.first_block) {              // the trailing CTAs of the launch
        trace_partial(trace.kstate, trace.G, trace.M, trace.K, (int)blockIdx.x - trace.first_block, trace.tr_part);
        return;
    }
    const unsigned per_chain = (unsigned)chain_rows_count<T, K>(lay);          // 32-bit index arithmetic (the launchers check the range)
    const unsigned total = per_chain * NCHAINS;
    const unsigned n_row_blocks = trace.kstate != nullptr ? (unsigned)trace.first_block : gridDim.x;
    for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += n_row_blocks * blockDim.x) {
        const unsigned chain = t / per_chain;
        const unsigned e = t - chain * per_chain;
        const ChainSpec<T>& sp = chain == 0 ? s0 : (chain == 1 ? s1 : (chain == 2 ? s2 : s3));
        out[t] = chain_rows_entry<T, K>(lay, sp, e);
    }
}

// Row tables of a batch (asvgp_elbo_grad_1d_batched): blockIdx.z = slot b, blockIdx.y = chain c of the slot — 0 the Kuu
// chain of Kuu[b], 2d+1 / 2d+2 the P chains (d/dl, d/dsigma2) of output column d — each table built with the matrix and
// right-hand-side functors of the single call (launch_kuu_chain, launch_pchains), so every entry has the same bits.
struct BatchRowsArgs {
    const double* Kuu; const double* dKuu;          // [B][K+1][M]
    const double* acc; size_t acc_stride;           // column d's packed accumulator at acc + d * acc_stride
    unsigned* counters; size_t counter_stride;      // finalize arrival counter of (b, d) at counters + (b * D + d) * counter_stride
    double inv_s2[ASVGP_MAX_BATCH], tan_s2[ASVGP_MAX_BATCH];   // 1 / sigma2 and -1 / sigma2^2 per slot (rounded on the host as there)
};
template <int K>
__global__ void __launch_bounds__(256) batch_rows_kernel(ChunkLayout lay, const __grid_constant__ BatchRowsArgs a, Dual<1>* __restrict__ out) {
    using T = Dual<1>;
    pdl_launch_dependents();
    const int M = lay.M, b = blockIdx.z, c = blockIdx.y, n_chains = gridDim.y;
    const size_t band = (size_t)(K + 1) * M;
    const double* Kuu = a.Kuu + b * band;
    const double* dKuu = a.dKuu + b * band;
    ChainSpec<T> sp{BandMat<T>{Kuu, dKuu, nullptr, 0.0, 0.0, 1, M}, VecRhs<T>{Kuu, M, 0}};
    if (c > 0) {
        const int d = (c - 1) >> 1;
        const double* G = a.acc + d * a.acc_stride;
        sp = (c & 1) ? ChainSpec<T>{BandMat<T>{Kuu, dKuu, G, a.inv_s2[b], 0.0, 1, M}, VecRhs<T>{G + band, M, 1}}
                     : ChainSpec<T>{BandMat<T>{Kuu, dKuu, G, a.inv_s2[b], a.tan_s2[b], 0, M}, VecRhs<T>{G + band, M, 1}};
        if ((c & 1) && blockIdx.x == 0 && threadIdx.x == 0) a.counters[((size_t)b * (n_chains >> 1) + d) * a.counter_stride] = 0u;
    }
    const unsigned per_chain = (unsigned)chain_rows_count<T, K>(lay);
    T* tab = out + ((size_t)b * n_chains + c) * per_chain;
    for (unsigned e = blockIdx.x * blockDim.x + threadIdx.x; e < per_chain; e += gridDim.x * blockDim.x)
        tab[e] = chain_rows_entry<T, K>(lay, sp, e);
}

// ------------------------------------------------------------------------------------------------------------------
// workspace carving (host) — one ChainWork per chain out of a caller-provided buffer
// ------------------------------------------------------------------------------------------------------------------
template <class T, int K>
struct ChainPlan {
    static size_t bytes(const ChunkLayout& lay) {
        const size_t n = ColumnStore<T, K, true>::count(lay.max_size(), lay.P) * sizeof(T);
        return (n + 255) & ~(size_t)255;
    }
    static ColumnStore<T, K, true> carve(const ChunkLayout& lay, char* base) {
        return ColumnStore<T, K, true>{reinterpret_cast<T*>(base), lay.max_size(), lay.P};
    }
};

// Shared-memory budget: the separator system, its factor and the per-chunk Schur pieces live in dynamic shared
// memory (they are touched by the single-thread phase, where global-memory latency would be fully exposed).
constexpr size_t kChainSmemLimit = 200 * 1024;

// One CTA = one chain.  `Mat`/`Rhs` feed the matrix; logdet/quad totals go to `tot`.
template <class T, int K, bool STORE, bool SOLVE, bool SELINV, class Mat, class Rhs, class Sink>
__device__ __forceinline__ void run_chain(const ChunkLayout& lay, const ColumnStore<T, K, true>& cols, char* smem,
                                          Mat A, Rhs rhs, T* x_out, Sink& sink, ChainTotals<T, K>* tot,
                                          long long* clk) {
    const int p = threadIdx.x;
    ChainWork<T, K> w;
    w.cols = cols;
    ChainSmall<T, K>::carve(lay.P, smem, w);
    if (p == 0 && clk) clk[0] = clock64();
    if (p < lay.P) chain_phase1<T, K, STORE>(lay, p, A, rhs, w);
    __syncthreads();
    if (p == 0 && clk) clk[1] = clock64();
    // separator system: block cyclic reduction, one lane per separator, two barriers per level (band_engine.cuh)
    const int n = lay.P - 1;
    if (p < n) cr_assemble<T, K>(lay, p, w);
    __syncthreads();
    for (int s = 1; s < n; s *= 2) {
        if (p < n && (p & (2 * s - 1)) == s) cr_eliminate<T, K>(n, s, p, lay.M, w);
        __syncthreads();
        if (p < n && (p & (2 * s - 1)) == 0) cr_update<T, K>(n, s, p, w);
        __syncthreads();
    }
    if (p == 0) {
        if (n > 0) cr_eliminate<T, K>(n, 0, 0, lay.M, w);
        *tot = chain_totals<T, K>(lay, w);
        if ((SOLVE || SELINV) && n > 0) cr_back<T, K, SOLVE, SELINV>(n, 0, 0, w);
    }
    __syncthreads();
    if ((SOLVE || SELINV) && n > 0) {
        for (int s = cr_top_stride(n); s >= 1; s /= 2) {
            if (p < n && (p & (2 * s - 1)) == s) cr_back<T, K, SOLVE, SELINV>(n, s, p, w);
            __syncthreads();
        }
        if (p < n) cr_export<T, K, SOLVE, SELINV>(lay, p, w);
        __syncthreads();
    }
    if (p == 0 && clk) clk[2] = clock64();
    if ((SOLVE || SELINV) && p < lay.P) chain_phase3<T, K, SOLVE, SELINV>(lay, p, w, x_out, sink);
    __syncthreads();
    if (p == 0 && clk) clk[3] = clock64();
}

// The same chain on a thread-block CLUSTER, with MORE LANES.  A lane's per-column cost is bound by its warp's fp64 issue
// slot (~250 fp64 instructions per column at one issue per two clocks: tools/chain_clocks.py — the per-column time does not
// change whether 128, 64 or 32 lanes share the SM), so the only way to shorten the sweeps is fewer columns per lane:
// P = 128 * n_cta chunks, CTA r sweeps chunks [128 r, 128 r + 128) with four full warps.  The separator system (P - 1 nodes)
// and the per-chunk Schur pieces are dealt over the CTAs' shared memories in the same way and reached through distributed
// shared memory (ChainWork::node / ::sch); the block cyclic reduction runs on all CTAs with cluster barriers between its
// levels; the reduced solution phase 3 reads goes through a small global scratch.
template <class T, int K, bool STORE, bool SOLVE, bool SELINV, class MakeMat, class MakeRhs, class MakeSink>
__device__ __forceinline__ void run_chain_cluster(const ChunkLayout& lay, const ColumnStore<T, K, true>& cols, char* smem, T* red_scratch,
                                                  MakeMat make_A, MakeRhs make_rhs, MakeSink make_sink, T* x_out,
                                                  ChainTotals<T, K>* tot, long long* clk) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank(), n_cta = (int)cluster.num_blocks();
    const int tid = threadIdx.x;
    const int per = kChainThreads;
    const int p = rank * per + tid;                               // this thread's chunk and separator node
    ChainWork<T, K> w;
    w.cols = cols;
    ChainSmall<T, K>::carve(per + 1, smem, w);                    // every CTA holds `per` Schur pieces and `per` nodes (carve(P) lays out P - 1 nodes)
    w.per_cta = per;
    const size_t nred = (size_t)lay.n_reduced();
    w.sig_red = red_scratch;
    w.x_red = red_scratch + (size_t)(2 * K) * nred;
#ifdef ASVGP_CHAIN_TRACE
    __shared__ long long s_trace[64];
    int n_trace = 0;
#define ASVGP_STAMP() do { if (rank == 0 && tid == 0 && n_trace < 64) s_trace[n_trace++] = clock64(); } while (0)
#else
#define ASVGP_STAMP() do {} while (0)
#endif
    cluster.sync();                                               // every CTA's shared memory exists before anybody writes to it
    ASVGP_STAMP();
    if (rank == 0 && tid == 0 && clk) clk[0] = clock64();
    if (p < lay.P) chain_phase1<T, K, STORE>(lay, p, make_A(p), make_rhs(p), w);
    cluster.sync();
    ASVGP_STAMP();
    if (rank == 0 && tid == 0 && clk) clk[1] = clock64();
    const int n = lay.P - 1;
    if (p < n) cr_assemble<T, K>(lay, p, w);
    cluster.sync();
    ASVGP_STAMP();
    for (int s = 1; s < n; s *= 2) {
        if (p < n && (p & (2 * s - 1)) == s) cr_eliminate<T, K>(n, s, p, lay.M, w);
        cluster.sync();
        ASVGP_STAMP();
        if (p < n && (p & (2 * s - 1)) == 0) cr_update<T, K>(n, s, p, w);
        cluster.sync();
        ASVGP_STAMP();
    }
    if (p == 0 && n > 0) cr_eliminate<T, K>(n, 0, 0, lay.M, w);
    cluster.sync();
    ASVGP_STAMP();
    {
        // totals: every lane brings its chunk's and its node's share; fixed-order tree inside the CTA, CTA partials added in rank order
        T ld = zero_of<T>(), qd = zero_of<T>();
        int info = 0;
        if (p < lay.P) { const ChunkSchur<T, K>& c = w.sch(p); ld += c.logdet; qd += c.quad; info = c.info; }
        if (p < n) { const CrNode<T, K>& nd = w.node(p); ld += nd.logdet; qd += nd.quad; if (info == 0) info = nd.info; }
        double v[4] = {value_of(ld), tangent_of(ld, 0), value_of(qd), tangent_of(qd, 0)};
        unsigned uinfo = info == 0 ? 0xffffffffu : (unsigned)info;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
            for (int i = 0; i < 4; ++i) v[i] += __shfl_xor_sync(0xffffffffu, v[i], o);
            uinfo = min(uinfo, __shfl_xor_sync(0xffffffffu, uinfo, o));
        }
        __shared__ double s_tot[kChainThreads / 32][4];
        __shared__ unsigned s_info[kChainThreads / 32];
        __shared__ double s_cta[5];
        if ((tid & 31) == 0) { for (int i = 0; i < 4; ++i) s_tot[tid >> 5][i] = v[i]; s_info[tid >> 5] = uinfo; }
        __syncthreads();
        if (tid == 0) {
            double a[4] = {0, 0, 0, 0};
            unsigned ui = 0xffffffffu;
            for (int wv = 0; wv < kChainThreads / 32; ++wv) { for (int i = 0; i < 4; ++i) a[i] += s_tot[wv][i]; ui = min(ui, s_info[wv]); }
            for (int i = 0; i < 4; ++i) s_cta[i] = a[i];
            s_cta[4] = (double)ui;
        }
        cluster.sync();
        ASVGP_STAMP();
        if (rank == 0 && tid == 0) {
            double a[4] = {0, 0, 0, 0};
            double ui = 4294967295.0;
            for (int r = 0; r < n_cta; ++r) {
                const double* q = cluster_peer(s_cta, r);
                for (int i = 0; i < 4; ++i) a[i] += q[i];
                ui = q[4] < ui ? q[4] : ui;
            }
            tot->logdet = make_scalar<T>(a[0], a[1]);
            tot->quad = make_scalar<T>(a[2], a[3]);
            tot->info = ui >= 4294967295.0 ? 0 : (int)ui;
        }
    }
    if ((SOLVE || SELINV) && n > 0) {
        if (p == 0) cr_back<T, K, SOLVE, SELINV>(n, 0, 0, w);
        cluster.sync();
        ASVGP_STAMP();
        for (int s = cr_top_stride(n); s >= 1; s /= 2) {
            if (p < n && (p & (2 * s - 1)) == s) cr_back<T, K, SOLVE, SELINV>(n, s, p, w);
            cluster.sync();
            ASVGP_STAMP();
        }
        if (p < n) cr_export<T, K, SOLVE, SELINV>(lay, p, w);
        __threadfence();
        cluster.sync();
        ASVGP_STAMP();
    }
    if (rank == 0 && tid == 0 && clk) clk[2] = clock64();
    if ((SOLVE || SELINV) && p < lay.P) {
        auto sink = make_sink(p);
        chain_phase3<T, K, SOLVE, SELINV>(lay, p, w, x_out, sink);
    }
    cluster.sync();                                               // nobody leaves while its shared memory may still be read
    ASVGP_STAMP();
    if (rank == 0 && tid == 0 && clk) clk[3] = clock64();
#ifdef ASVGP_CHAIN_TRACE
    if (rank == 0 && tid == 0) {
        for (int i = 1; i < n_trace; ++i) printf("trace blk=%d SELINV=%d P=%d step=%d %lld\n", (int)blockIdx.x, (int)SELINV, lay.P, i, s_trace[i] - s_trace[i - 1]);
    }
#endif
#undef ASVGP_STAMP
}

// ------------------------------------------------------------------------------------------------------------------
// ELBO + gradient
// ------------------------------------------------------------------------------------------------------------------
// The ELBO's work is split where its data dependencies are (DESIGN.md §4.2):
//   Kuu chain  (chain 0: [Kuu, d/dl], factorisation + Takahashi) depends on the hyper-parameters only.  It leaves
//              log|Kuu|, its tangent and band(Kuu^-1) (value + tangent) in a small "Kuu state" buffer — and can therefore
//              run on a side stream WHILE the O(N) accumulate produces G (asvgp_kuu_chain_1d);
//   P chains   (chains 1, 2: [P, d/dl], [P, d/dsigma2], forward only) need G and b;
//   finalize   trace(Kuu^-1 G) = sum band(Kuu^-1) .* band(G) (off-diagonals twice, reference gpr.py:60-70) as a fixed-order
//              dot product of the stored inverse band with G, then the bound and its derivatives.
// per-launch record area: [2][16] chain records, the finalize kernel's arrival counter (double slot 32), the [kTraceBlocks][2]
// trace partials (from slot 64); one per output column of every slot in a batch
constexpr size_t kPartialBytes = 2048, kPartialDoubles = kPartialBytes / sizeof(double);

// Chains of every slot of a batch (blockIdx.y; one slot outside asvgp_elbo_grad_1d_batched) in one launch.  Chain c of a slot is
// 0: the Kuu chain;  2d+1: P of output column d with tangent d/dl;  2d+2: the same P with tangent d/dsigma2.
// A launch runs chains first_chain .. first_chain + n_chains - 1 of each slot, launched chain i = slot * n_chains + (c - first_chain).
template <int K>
struct ElboArgs {
    ChunkLayout lay;
    int first_chain, n_chains;
    char* cols; size_t cols_bytes;          // launched chain i's column store at cols + i * cols_bytes
    const Dual<1>* rows;                    // and its lane-interleaved row table at rows + i * chain_rows_count
    Dual<1>* red_scratch;                   // and its reduced-solution scratch at red_scratch + i * red_scratch_count (clusters)
    double* kstate; size_t kstate_stride;   // slot's Kuu state: the Kuu chain's [16] record, then band(Kuu^-1) (K+1) x M duals
    double* partial; size_t partial_stride; // slot's P-chain records ([16]: logdet, dlogdet, quad, dquad, -, -, info, -, clocks[4]):
                                            // column d at partial + slot * partial_stride + d * kPartialDoubles, + 16 for d/dsigma2
    __device__ __forceinline__ int launched(int slot, int c) const { return slot * n_chains + c; }
    __device__ __forceinline__ double* record(int slot, int chain) const {
        if (chain == 0) return kstate + slot * kstate_stride;
        return partial + slot * partial_stride + ((chain - 1) >> 1) * kPartialDoubles + 16 * ((chain - 1) & 1);
    }
    __device__ __forceinline__ Dual<1>* kinv(int slot) const { return reinterpret_cast<Dual<1>*>(kstate + slot * kstate_stride + 16); }
};
template <class T, int K>
__device__ __forceinline__ ColumnStore<T, K, true> launched_cols(const ChunkLayout& lay, char* cols, size_t cols_bytes, int i) {
    return ColumnStore<T, K, true>{reinterpret_cast<T*>(cols + (size_t)i * cols_bytes), lay.max_size(), lay.P};
}

template <int K>
__global__ void __launch_bounds__(kChainThreads) elbo_chains_kernel(ElboArgs<K> a) {
    using T = Dual<1>;
    extern __shared__ __align__(16) char smem[];
    const int slot = blockIdx.y, chain = a.first_chain + blockIdx.x, li = a.launched(slot, blockIdx.x), p = threadIdx.x;
    const ChunkLayout lay = a.lay;
    const int M = lay.M;
    __shared__ ChainTotals<T, K> tot;
    __shared__ long long clk[4];
    double* out = a.record(slot, chain);
    const ColumnStore<T, K, true> cols = launched_cols<T, K>(lay, a.cols, a.cols_bytes, li);
    pdl_launch_dependents();
    pdl_wait();                              // the row tables are complete

    const int n_rho = chain_n_rho(lay, K), g0 = lay.P > 1 ? lay.start(p < lay.P ? p : 0) : 0, pp = p < lay.P ? p : 0;
    const T* tab = a.rows + (size_t)li * chain_rows_count<T, K>(lay);
    const RowsMat<T, K> A{tab, g0, lay.P, pp, n_rho};
    const RowsRhs<T> rhs{tab + (size_t)n_rho * (K + 1) * lay.P, g0, lay.P, pp, n_rho};
    if (chain == 0) {
        BandSink<T> sink{a.kinv(slot), M};
        run_chain<T, K, true, false, true>(lay, cols, smem, A, rhs, static_cast<T*>(nullptr), sink, &tot, clk);
    } else {
        // P with tangent d/dl or d/dsigma2 (tables built by the launcher)
        BandSink<T> no_sink{nullptr, M};
        run_chain<T, K, false, false, false>(lay, cols, smem, A, rhs, static_cast<T*>(nullptr), no_sink, &tot, clk);
    }
    if (p == 0) {
        out[0] = tot.logdet.v; out[1] = tot.logdet.d[0];
        out[2] = tot.quad.v;   out[3] = tot.quad.d[0];
        out[6] = (double)tot.info;
        const long long t_end = clock64();
        out[8] = (double)(clk[1] - clk[0]); out[9] = (double)(clk[2] - clk[1]);
        out[10] = (double)(clk[3] - clk[2]); out[11] = (double)(t_end - clk[3]);
    }
}

// Cluster version (M large): launched chain `slot` runs on cluster `slot` of NCTA CTAs with 128 * NCTA chunks.
template <int K, int NCTA>
__global__ void __cluster_dims__(NCTA, 1, 1) __launch_bounds__(kChainThreads) elbo_chains_cluster_kernel(ElboArgs<K> a) {
    using T = Dual<1>;
    extern __shared__ __align__(16) char smem[];
    const int slot = blockIdx.y, c = blockIdx.x / NCTA, chain = a.first_chain + c, li = a.launched(slot, c);
    const int rank = blockIdx.x % NCTA, tid = threadIdx.x;
    const ChunkLayout lay = a.lay;
    __shared__ ChainTotals<T, K> tot;
    __shared__ long long clk[4];
    double* out = a.record(slot, chain);
    const ColumnStore<T, K, true> cols = launched_cols<T, K>(lay, a.cols, a.cols_bytes, li);
    pdl_launch_dependents();
    pdl_wait();                              // the row tables are complete
    const int n_rho = chain_n_rho(lay, K);
    const T* tab = a.rows + (size_t)li * chain_rows_count<T, K>(lay);
    T* scratch = a.red_scratch + (size_t)li * ((size_t)(2 * K + 1) * lay.n_reduced() + 8);
    auto g0_of = [&](int lane) { return lay.P > 1 ? lay.start(lane) : 0; };
    auto make_A = [&](int lane) { return RowsMat<T, K>{tab, g0_of(lane), lay.P, lane, n_rho}; };
    auto make_rhs = [&](int lane) { return RowsRhs<T>{tab + (size_t)n_rho * (K + 1) * lay.P, g0_of(lane), lay.P, lane, n_rho}; };
    if (chain == 0) {
        auto make_sink = [&](int) { return BandSink<T>{a.kinv(slot), lay.M}; };
        run_chain_cluster<T, K, true, false, true>(lay, cols, smem, scratch, make_A, make_rhs, make_sink, static_cast<T*>(nullptr), &tot, clk);
    } else {
        auto make_sink = [&](int) { return BandSink<T>{nullptr, lay.M}; };
        run_chain_cluster<T, K, false, false, false>(lay, cols, smem, scratch, make_A, make_rhs, make_sink, static_cast<T*>(nullptr), &tot, clk);
    }
    if (rank == 0 && tid == 0) {
        out[0] = tot.logdet.v; out[1] = tot.logdet.d[0];
        out[2] = tot.quad.v;   out[3] = tot.quad.d[0];
        out[6] = (double)tot.info;
        const long long t_end = clock64();
        out[8] = (double)(clk[1] - clk[0]); out[9] = (double)(clk[2] - clk[1]);
        out[10] = (double)(clk[3] - clk[2]); out[11] = (double)(t_end - clk[3]);
    }
}

// Collapsed bound of reference gpr.py:81-87 and its derivatives.  With Q = b^T P^-1 b (so that
// sum(c^2) = Q / sigma2^2, gpr.py:75,85), tr = trace(Kuu^-1 G):
//   ELBO = -N/2 log(2 pi s2) - 1/2 log|P| + 1/2 log|Kuu| - yy/(2 s2) + Q/(2 s2^2) - N v/(2 s2) + tr/(2 s2)
// Kuu = Kt(l)/v  =>  P = (Kt + (v/s2) G)/v, hence d/dv of log|P| and Q follow from d/ds2:
//   dlog|P|/dv = -M/v - (s2/v) dlog|P|/ds2,   dQ/dv = Q/v - (s2/v) dQ/ds2,   dlog|Kuu|/dv = -M/v,   dtr/dv = tr/v.
// trace_done = 0: launched with kTraceBlocks CTAs that compute the trace partials first (trace_partial); the CTA that arrives
// last combines.  trace_done = 1: the partials are there already (the P chains' chain_rows_kernel hosted the trace CTAs), one CTA.
// One bound: `block` is this CTA's trace share (trace_done = 0, kTraceBlocks CTAs per bound), the sums are the same whichever
// CTA arrives last.
__device__ __forceinline__ void elbo_finalize(const double* __restrict__ kstate, double* __restrict__ partial,
                                              const double* __restrict__ G, const double* __restrict__ scal,
                                              int M, int K, double variance, double sigma2, int trace_done, int block,
                                              double* __restrict__ out) {
    double* tr_part = partial + 64;                                     // [kTraceBlocks][2]
    unsigned* counter = reinterpret_cast<unsigned*>(partial + 32);      // zeroed by the P chains' row-table kernel
    if (!trace_done) {
        trace_partial(kstate, G, M, K, block, tr_part);
        if (threadIdx.x != 0) return;
        __threadfence();
        if (atomicAdd(counter, 1u) != kTraceBlocks - 1) return;
        __threadfence();
    } else if (threadIdx.x != 0) {
        return;
    }
    double tr = 0.0, dtr_dl = 0.0;
    for (int i = 0; i < kTraceBlocks; ++i) { tr += __ldcg(tr_part + 2 * i); dtr_dl += __ldcg(tr_part + 2 * i + 1); }
    const double* cK = kstate;           // Kuu chain (d/dl)
    const double* cL = partial;          // P chain (d/dl)
    const double* cS = partial + 16;     // P chain (d/dsigma2)
    const double yy = scal[0], N = scal[1];
    const double v = variance, s2 = sigma2;
    const double logdetK = cK[0], dlogdetK_dl = cK[1];
    const double logdetP = cL[0], dlogdetP_dl = cL[1], Q = cL[2], dQ_dl = cL[3];
    const double dlogdetP_ds = cS[1], dQ_ds = cS[3];
    const double two_pi = 6.283185307179586476925286766559;
    const double elbo = -0.5 * N * log(two_pi * s2) - 0.5 * logdetP + 0.5 * logdetK - 0.5 * yy / s2
                        + 0.5 * Q / (s2 * s2) - 0.5 * N * v / s2 + 0.5 * tr / s2;
    const double d_l = -0.5 * dlogdetP_dl + 0.5 * dlogdetK_dl + 0.5 * dQ_dl / (s2 * s2) + 0.5 * dtr_dl / s2;
    const double d_s = -0.5 * N / s2 - 0.5 * dlogdetP_ds + 0.5 * yy / (s2 * s2) + 0.5 * dQ_ds / (s2 * s2)
                       - Q / (s2 * s2 * s2) + 0.5 * N * v / (s2 * s2) - 0.5 * tr / (s2 * s2);
    const double dlogdetP_dv = -(double)M / v - (s2 / v) * dlogdetP_ds;
    const double dQ_dv = Q / v - (s2 / v) * dQ_ds;
    const double d_v = -0.5 * dlogdetP_dv - 0.5 * (double)M / v + 0.5 * dQ_dv / (s2 * s2) - 0.5 * N / s2
                       + 0.5 * tr / (v * s2);
    out[0] = elbo; out[1] = d_v; out[2] = d_l; out[3] = d_s;
    out[4] = logdetK; out[5] = logdetP; out[6] = Q; out[7] = tr;
    double info = cK[6];
    if (info == 0.0) info = cL[6];
    if (info == 0.0) info = cS[6];
    out[8] = info;
    // diagnostics: SM cycles of the Kuu chain's phases (chunk sweep, separator system, back sweep, tail)
    out[9] = cK[8]; out[10] = cK[9]; out[11] = cK[10]; out[12] = cK[11];
    out[13] = cL[8]; out[14] = cL[9];
    out[15] = dtr_dl;             // d trace(Kuu^-1 G) / d lengthscale (multi-output bound: trace terms count once)
}

__global__ void __launch_bounds__(kTraceThreads) elbo_finalize_kernel(const double* __restrict__ kstate, double* __restrict__ partial,
                                                                      const double* __restrict__ G, const double* __restrict__ scal,
                                                                      int M, int K, double variance, double sigma2, int trace_done,
                                                                      double* __restrict__ out) {
    pdl_wait();                                                         // the P chains are complete
    elbo_finalize(kstate, partial, G, scal, M, K, variance, sigma2, trace_done, (int)blockIdx.x, out);
}

// The bounds of a batch: blockIdx.z = slot b, blockIdx.y = output column d, kTraceBlocks CTAs each; out[b][d][16].
struct BatchFinalizeArgs {
    const double* kstate; size_t kstate_stride;
    double* partial; size_t partial_stride;          // as ElboArgs
    const double* acc; size_t acc_stride;
    double variance[ASVGP_MAX_BATCH], sigma2[ASVGP_MAX_BATCH];
};
__global__ void __launch_bounds__(kTraceThreads) elbo_finalize_batched_kernel(const __grid_constant__ BatchFinalizeArgs a, int M, int K,
                                                                              double* __restrict__ out) {
    pdl_wait();                                                         // every chain of the batch is complete
    const int b = blockIdx.z, d = blockIdx.y, D = gridDim.y;
    const double* G = a.acc + d * a.acc_stride;
    elbo_finalize(a.kstate + b * a.kstate_stride, a.partial + b * a.partial_stride + d * kPartialDoubles, G, G + (size_t)(K + 2) * M,
                  M, K, a.variance[b], a.sigma2[b], 0, (int)blockIdx.x, out + ((size_t)b * D + d) * 16);
}

// ------------------------------------------------------------------------------------------------------------------
// posterior weights
// ------------------------------------------------------------------------------------------------------------------
template <int K>
struct PosteriorArgs {
    ChunkLayout lay;
    ColumnStore<double, K, true> cols[2];
    const double* Kuu; const double* G; const double* b;
    double sigma2;
    double* sigK; double* sigP; double* x;       // (K+1) x M, (K+1) x M, M
    double* info;                                // [2]
    const double* rows;                          // lane-interleaved row tables of the two chains
};

template <int K>
__global__ void __launch_bounds__(kChainThreads) posterior_chains_kernel(PosteriorArgs<K> a) {
    using T = double;
    extern __shared__ __align__(16) char smem[];
    const int chain = blockIdx.x, p = threadIdx.x;
    const ChunkLayout lay = a.lay;
    const int M = lay.M;
    __shared__ ChainTotals<T, K> tot;
    (void)M;
    const int n_rho = chain_n_rho(lay, K), g0 = lay.P > 1 ? lay.start(p < lay.P ? p : 0) : 0, pp = p < lay.P ? p : 0;
    const T* tab = a.rows + (size_t)chain * chain_rows_count<T, K>(lay);
    const RowsMat<T, K> A{tab, g0, lay.P, pp, n_rho};
    const RowsRhs<T> rhs{tab + (size_t)n_rho * (K + 1) * lay.P, g0, lay.P, pp, n_rho};
    BandSink<T> sinkK{a.sigK, lay.M}, sinkP{a.sigP, lay.M};
    if (chain == 0) run_chain<T, K, true, false, true>(lay, a.cols[0], smem, A, rhs, static_cast<T*>(nullptr), sinkK, &tot, nullptr);
    else run_chain<T, K, true, true, true>(lay, a.cols[1], smem, A, rhs, a.x, sinkP, &tot, nullptr);
    if (p == 0) a.info[chain] = (double)tot.info;
}

__global__ void __launch_bounds__(256) posterior_combine_kernel(const double* __restrict__ sigK,
                                                                const double* __restrict__ sigP,
                                                                const double* __restrict__ x, double inv_s2, int M,
                                                                int band_elems, double* __restrict__ alpha,
                                                                double* __restrict__ S) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < band_elems; i += gridDim.x * blockDim.x) {
        S[i] = sigP[i] - sigK[i];
        if (i < M) alpha[i] = x[i] * inv_s2;
    }
}


// ------------------------------------------------------------------------------------------------------------------
// band(A^-1) and log|A| of one SPD band matrix with one tangent — used for the per-dimension factors K1, K2 of the
// Kronecker model (log|K1 (x) K2| = m2 log|K1| + m1 log|K2| and trace((K1 (x) K2)^-1 G) only need the bands of the
// factor inverses, reference gpr.py:288-289,307)
// ------------------------------------------------------------------------------------------------------------------
template <int K>
struct BandInvArgs {
    ChunkLayout lay;
    ColumnStore<Dual<1>, K, true> cols;
    const double* A; const double* dA;
    Dual<1>* sig;             // scratch (K+1) x M duals
    double* sig_val; double* sig_tan;
    double* scal;             // [4]: log|A|, d log|A|, info, -
    const Dual<1>* rows;      // lane-interleaved row table
};

template <int K>
__global__ void __launch_bounds__(kChainThreads) band_inverse_kernel(BandInvArgs<K> a) {
    using T = Dual<1>;
    extern __shared__ __align__(16) char smem[];
    const int p = threadIdx.x;
    const ChunkLayout lay = a.lay;
    const int M = lay.M;
    __shared__ ChainTotals<T, K> tot;
    const int n_rho = chain_n_rho(lay, K), g0 = lay.P > 1 ? lay.start(p < lay.P ? p : 0) : 0, pp = p < lay.P ? p : 0;
    const RowsMat<T, K> A{a.rows, g0, lay.P, pp, n_rho};
    const RowsRhs<T> rhs{a.rows + (size_t)n_rho * (K + 1) * lay.P, g0, lay.P, pp, n_rho};
    BandSink<T> sink{a.sig, lay.M};
    run_chain<T, K, true, false, true>(lay, a.cols, smem, A, rhs, static_cast<T*>(nullptr), sink, &tot, nullptr);
    for (int i = p; i < (K + 1) * M; i += kChainThreads) {
        const T s = a.sig[i];
        a.sig_val[i] = s.v;
        a.sig_tan[i] = s.d[0];
    }
    if (p == 0) {
        a.scal[0] = tot.logdet.v; a.scal[1] = tot.logdet.d[0]; a.scal[2] = (double)tot.info; a.scal[3] = 0.0;
    }
}

template <int K>
static int launch_band_inverse(const ChunkLayout& lay, const double* A, const double* dA, double* sig_val,
                               double* sig_tan, double* scal, char* work, cudaStream_t st) {
    BandInvArgs<K> a;
    a.lay = lay;
    char* p = work;
    a.cols = ChainPlan<Dual<1>, K>::carve(lay, p);
    p += ChainPlan<Dual<1>, K>::bytes(lay);
    a.sig = reinterpret_cast<Dual<1>*>(p);
    a.A = A; a.dA = dA; a.sig_val = sig_val; a.sig_tan = sig_tan; a.scal = scal;
    p += ((size_t)(K + 1) * lay.M * sizeof(Dual<1>) + 255) & ~(size_t)255;
    Dual<1>* rows = reinterpret_cast<Dual<1>*>(p);
    a.rows = rows;
    {
        using T = Dual<1>;
        ChainSpec<T> s0{BandMat<T>{A, dA, nullptr, 0.0, 0.0, 1, lay.M}, VecRhs<T>{A, lay.M, 0}};
        const size_t total = chain_rows_count<T, K>(lay);
        chain_rows_kernel<T, K, 1><<<(int)((total + 255) / 256), 256, 0, st>>>(lay, s0, s0, s0, s0, rows); ASVGP_LAUNCHED();
        ASVGP_CUDA_OK(cudaGetLastError());
    }
    ASVGP_CUDA_OK(cudaMemsetAsync(a.sig, 0, (size_t)(K + 1) * lay.M * sizeof(Dual<1>), st));
    const size_t smem = ChainSmall<Dual<1>, K>::bytes(lay.P);
    ASVGP_CUDA_OK(cudaFuncSetAttribute(band_inverse_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    band_inverse_kernel<K><<<1, kChainThreads, smem, st>>>(a); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

static size_t align256(size_t n) { return (n + 255) & ~(size_t)255; }
// Programmatic dependent launch: the kernel may be scheduled while its predecessor in the stream is still running (its CTAs
// park in pdl_wait() until that grid has completed and flushed), which takes the launch latency and the cluster's
// co-scheduling off the chain of three dependent launches (row tables -> chains -> bound).
template <class... KArgs, class... Args>
static cudaError_t launch_dependent(void (*kernel)(KArgs...), dim3 grid, int block, size_t smem, cudaStream_t st, bool pdl, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
// cudaFuncAttributeMaxDynamicSharedMemorySize, set once per kernel and size (the call costs host time on every launch otherwise)
template <class Kernel>
static cudaError_t allow_smem(Kernel kernel, size_t smem) {
    static size_t allowed = 0;          // one per kernel type = per instantiation
    static const void* which = nullptr;
    if (which == reinterpret_cast<const void*>(kernel) && smem <= allowed) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) { allowed = smem; which = reinterpret_cast<const void*>(kernel); }
    return e;
}
template <int K>
static size_t red_scratch_count(const ChunkLayout& lay) { return (size_t)(2 * K + 1) * lay.n_reduced() + 8; }     // per chain (clustered layout)
// workspace of one launch of n_chains chains: column stores, [n_chains][16] partials, row tables, reduced-solution scratch
template <int K>
static size_t chains_work_bytes(const ChunkLayout& lay, int n_chains) {
    return n_chains * ChainPlan<Dual<1>, K>::bytes(lay) + kPartialBytes + align256(n_chains * chain_rows_count<Dual<1>, K>(lay) * sizeof(Dual<1>))
           + align256(n_chains * red_scratch_count<K>(lay) * sizeof(Dual<1>));
}
static size_t kuu_state_doubles(int M, int K) { return 16 + 2 * (size_t)(K + 1) * M; }
template <int K>
static size_t elbo_work_bytes(const ChunkLayout& lay) {
    return chains_work_bytes<K>(lay, 1) + chains_work_bytes<K>(lay, 2) + align256(kuu_state_doubles(lay.M, K) * sizeof(double));
}
template <int K>
static size_t posterior_work_bytes(const ChunkLayout& lay) {
    return 2 * ChainPlan<double, K>::bytes(lay) + 3 * ((((size_t)(K + 1) * lay.M * sizeof(double)) + 255) & ~(size_t)255)
           + 256 + (((size_t)lay.M * sizeof(double) + 255) & ~(size_t)255) + 2 * chain_rows_count<double, K>(lay) * sizeof(double) + 256;
}

// The chain kernel of `a` for `n_slots` slots (blockIdx.y): one CTA per chain, or a cluster of lay.P / 128 CTAs
// (pick_layout_elbo).  smem_floor: see launch_chain_group.
template <int K>
static int launch_chains(const ElboArgs<K>& a, int n_slots, size_t smem_floor, bool pdl, cudaStream_t st) {
    using T = Dual<1>;
    const ChunkLayout& lay = a.lay;
    const int n_cta = (lay.P + kChainThreads - 1) / kChainThreads;          // > 1: clustered layout
    if (n_cta > 1) {
        const size_t smem = std::max(ChainSmall<T, K>::bytes(kChainThreads + 1), smem_floor);
        const dim3 grid(a.n_chains * n_cta, n_slots);
        if (n_cta == 2) {
            ASVGP_CUDA_OK(allow_smem(elbo_chains_cluster_kernel<K, 2>, smem));
            ASVGP_CUDA_OK(launch_dependent(elbo_chains_cluster_kernel<K, 2>, grid, kChainThreads, smem, st, pdl, a));
        } else if (n_cta == 8) {
            ASVGP_CUDA_OK(allow_smem(elbo_chains_cluster_kernel<K, 8>, smem));
            ASVGP_CUDA_OK(launch_dependent(elbo_chains_cluster_kernel<K, 8>, grid, kChainThreads, smem, st, pdl, a));
        } else {
            ASVGP_CUDA_OK(allow_smem(elbo_chains_cluster_kernel<K, 4>, smem));
            ASVGP_CUDA_OK(launch_dependent(elbo_chains_cluster_kernel<K, 4>, grid, kChainThreads, smem, st, pdl, a));
        }
    } else {
        const size_t smem = std::max(ChainSmall<T, K>::bytes(lay.P), smem_floor);
        ASVGP_CUDA_OK(allow_smem(elbo_chains_kernel<K>, smem));
        ASVGP_CUDA_OK(launch_dependent(elbo_chains_kernel<K>, dim3(a.n_chains, n_slots), kChainThreads, smem, st, pdl, a));
    }
    ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

// Row tables + chain kernel of `n_chains` chains starting at chain `first_chain` (0: Kuu; 1, 2: P with d/dl, d/dsigma2).
// `kstate` receives the Kuu chain's record and band(Kuu^-1); returns the P chains' partials in work.
template <int K>
static int launch_chain_group(const ChunkLayout& lay, int first_chain, int n_chains, const ChainSpec<Dual<1>>& s0,
                              const ChainSpec<Dual<1>>& s1, double* kstate, char* work, double** partials_out,
                              cudaEvent_t gate, TraceJob trace, cudaStream_t st) {
    using T = Dual<1>;
    ElboArgs<K> a;
    a.lay = lay;
    a.first_chain = first_chain;
    a.n_chains = n_chains;
    char* p = work;
    a.cols = p;
    a.cols_bytes = ChainPlan<T, K>::bytes(lay);
    p += n_chains * a.cols_bytes;
    double* partial = reinterpret_cast<double*>(p);
    p += kPartialBytes;
    a.kstate = kstate;
    a.kstate_stride = 0;
    a.partial = partial;
    a.partial_stride = 0;
    if (partials_out != nullptr) *partials_out = partial;
    T* rows = reinterpret_cast<T*>(p);
    p += align256(n_chains * chain_rows_count<T, K>(lay) * sizeof(T));
    a.rows = rows;
    a.red_scratch = reinterpret_cast<T*>(p);
    const size_t total = n_chains * chain_rows_count<T, K>(lay);
    ASVGP_REQUIRE(total < ((size_t)1 << 31), "banded chains: %zu row-table entries exceed the 32-bit index range", total);
    const int grid = (int)std::min<size_t>((total + 255) / 256, 148 * 8);
    if (n_chains == 1) {
        chain_rows_kernel<T, K, 1><<<grid, 256, 0, st>>>(lay, s0, s0, s0, s0, rows);
    } else {
        trace.first_block = grid;
        trace.tr_part = partial + 64;
        chain_rows_kernel<T, K, 2><<<grid + (trace.kstate != nullptr ? kTraceBlocks : 0), 256, 0, st>>>(
            lay, s0, s1, s1, s1, rows, reinterpret_cast<unsigned*>(partial + 32), trace);
    }
    ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    if (gate != nullptr) ASVGP_CUDA_OK(cudaEventRecord(gate, st));          // "the chain kernel is next in line"
    // A gated chain runs BESIDE a streaming kernel whose CTAs all carry the same share of the work: one of them landing on a
    // chain SM (shared issue slots, the L1 invalidation of every cluster barrier) becomes the straggler the whole kernel waits
    // for (+12 % on the accumulate, measured).  Asking for all of the SM's shared memory keeps the chain's SMs to itself.
    const size_t smem_floor = gate != nullptr ? (size_t)(227 * 1024 - 2048) : 0;
    // an event record between the two launches rules the early launch out
    return launch_chains<K>(a, 1, smem_floor, gate == nullptr, st);
}

// The Kuu chain: log|Kuu|, its d/dl and band(Kuu^-1) with tangent into `kstate` ([16] record + (K+1) x M duals).
template <int K>
static int launch_kuu_chain(const ChunkLayout& lay, const double* Kuu, const double* dKuu, double* kstate, char* work, cudaEvent_t gate,
                            cudaStream_t st) {
    using T = Dual<1>;
    const int M = lay.M;
    ChainSpec<T> s0{BandMat<T>{Kuu, dKuu, nullptr, 0.0, 0.0, 1, M}, VecRhs<T>{Kuu, M, 0}};
    return launch_chain_group<K>(lay, 0, 1, s0, s0, kstate, work, nullptr, gate, TraceJob{nullptr, nullptr, nullptr, 0, 0, 0}, st);
}

// The two P chains and the bound, given the Kuu state.
template <int K>
static int launch_pchains(const ChunkLayout& lay, const double* kstate, const double* Kuu, const double* dKuu, const double* acc,
                          double variance, double sigma2, double* out, char* work, cudaEvent_t kuu_ready, int join_late, cudaStream_t st) {
    using T = Dual<1>;
    const int M = lay.M;
    const double* G = acc;
    const double* b = acc + (size_t)(K + 1) * M;
    const double inv_s2 = 1.0 / sigma2;
    // chain 1: P = Kuu + G/s2 with d/dl;  chain 2: P with d/dsigma2 = -G/s2^2
    ChainSpec<T> s1{BandMat<T>{Kuu, dKuu, G, inv_s2, 0.0, 1, M}, VecRhs<T>{b, M, 1}};
    ChainSpec<T> s2{BandMat<T>{Kuu, dKuu, G, inv_s2, -inv_s2 * inv_s2, 0, M}, VecRhs<T>{b, M, 1}};
    double* partial = nullptr;
    // join_late = 0: the Kuu state is (about to be) complete — join first and let the row-table launch host the trace CTAs;
    // join_late = 1: the Kuu chain may still be running beside us — join only where its state is first read, after the P chains.
    if (!join_late && kuu_ready != nullptr) ASVGP_CUDA_OK(cudaStreamWaitEvent(st, kuu_ready, 0));
    const TraceJob trace{join_late ? nullptr : kstate, G, nullptr, M, K, 0};
    if (int rc = launch_chain_group<K>(lay, 1, 2, s1, s2, nullptr, work, &partial, nullptr, trace, st)) return rc;
    if (join_late && kuu_ready != nullptr) ASVGP_CUDA_OK(cudaStreamWaitEvent(st, kuu_ready, 0));
    const bool pdl = !(join_late && kuu_ready != nullptr);       // nothing between the chain kernel and this launch
    ASVGP_CUDA_OK(launch_dependent(elbo_finalize_kernel, join_late ? kTraceBlocks : 1, kTraceThreads, 0, st, pdl, kstate, partial, G,
                                   acc + (size_t)(K + 2) * M, M, K, variance, sigma2, join_late ? 0 : 1, out));
    ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

template <int K>
static int launch_elbo(const ChunkLayout& lay, const double* Kuu, const double* dKuu, const double* acc,
                       double variance, double sigma2, double* out, char* work, cudaStream_t st) {
    double* kstate = reinterpret_cast<double*>(work + chains_work_bytes<K>(lay, 1));
    char* pwork = work + chains_work_bytes<K>(lay, 1) + align256(kuu_state_doubles(lay.M, K) * sizeof(double));
    if (int rc = launch_kuu_chain<K>(lay, Kuu, dKuu, kstate, work, nullptr, st)) return rc;
    return launch_pchains<K>(lay, kstate, Kuu, dKuu, acc, variance, sigma2, out, pwork, nullptr, 0, st);
}

// Workspace of a batch of B slots with D output columns: per chain (B (1 + 2D) of them) a column store, a row table and
// reduced-solution scratch; per slot a Kuu state; per (slot, column) a record area.
template <int K>
struct BatchPlan {
    size_t cols_bytes, rows_off, scratch_off, kstate_off, kstate_stride, partial_off, total;
    BatchPlan(const ChunkLayout& lay, int B, int D) {
        const size_t n = (size_t)B * (1 + 2 * D);
        cols_bytes = ChainPlan<Dual<1>, K>::bytes(lay);
        rows_off = n * cols_bytes;
        scratch_off = rows_off + align256(n * chain_rows_count<Dual<1>, K>(lay) * sizeof(Dual<1>));
        kstate_off = scratch_off + align256(n * red_scratch_count<K>(lay) * sizeof(Dual<1>));
        kstate_stride = align256(kuu_state_doubles(lay.M, K) * sizeof(double)) / sizeof(double);
        partial_off = kstate_off + (size_t)B * kstate_stride * sizeof(double);
        total = partial_off + (size_t)B * D * kPartialBytes;
    }
};

// B bounds with D output columns each in three launches: the row tables of every chain, every chain (the Kuu chains beside the
// P chains: these read Kuu, not the Kuu state), the trace and the bound of every (slot, column).  Each chain, trace share and
// bound runs the code of the single call on its own workspace, so slot b's bits depend neither on B nor on the other slots.
template <int K>
static int launch_elbo_batched(const ChunkLayout& lay, int B, int D, const double* Kuu, const double* dKuu, const double* acc,
                               const double* h_variance, const double* h_sigma2, double* out, char* work, cudaStream_t st) {
    using T = Dual<1>;
    const BatchPlan<K> plan(lay, B, D);
    const int M = lay.M;
    const size_t acc_stride = (size_t)(K + 2) * M + 2;
    const size_t per_chain = chain_rows_count<T, K>(lay);
    ASVGP_REQUIRE(per_chain < ((size_t)1 << 31), "banded chains: %zu row-table entries exceed the 32-bit index range", per_chain);
    ElboArgs<K> a;
    a.lay = lay;
    a.first_chain = 0;
    a.n_chains = 1 + 2 * D;
    a.cols = work;
    a.cols_bytes = plan.cols_bytes;
    a.rows = reinterpret_cast<T*>(work + plan.rows_off);
    a.red_scratch = reinterpret_cast<T*>(work + plan.scratch_off);
    a.kstate = reinterpret_cast<double*>(work + plan.kstate_off);
    a.kstate_stride = plan.kstate_stride;
    a.partial = reinterpret_cast<double*>(work + plan.partial_off);
    a.partial_stride = (size_t)D * kPartialDoubles;

    BatchRowsArgs r;
    r.Kuu = Kuu; r.dKuu = dKuu; r.acc = acc; r.acc_stride = acc_stride;
    r.counters = reinterpret_cast<unsigned*>(a.partial + 32);
    r.counter_stride = kPartialBytes / sizeof(unsigned);
    for (int b = 0; b < B; ++b) {
        const double inv_s2 = 1.0 / h_sigma2[b];       // as launch_pchains
        r.inv_s2[b] = inv_s2;
        r.tan_s2[b] = -inv_s2 * inv_s2;
    }
    const int n_tables = a.n_chains * B;
    const int gx = (int)std::min<size_t>((per_chain + 255) / 256, std::max(1, 148 * 8 / n_tables));
    batch_rows_kernel<K><<<dim3(gx, a.n_chains, B), 256, 0, st>>>(lay, r, reinterpret_cast<T*>(work + plan.rows_off)); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    if (int rc = launch_chains<K>(a, B, 0, true, st)) return rc;
    BatchFinalizeArgs f;
    f.kstate = a.kstate; f.kstate_stride = a.kstate_stride;
    f.partial = a.partial; f.partial_stride = a.partial_stride;
    f.acc = acc; f.acc_stride = acc_stride;
    for (int b = 0; b < B; ++b) { f.variance[b] = h_variance[b]; f.sigma2[b] = h_sigma2[b]; }
    ASVGP_CUDA_OK(launch_dependent(elbo_finalize_batched_kernel, dim3(kTraceBlocks, D, B), kTraceThreads, 0, st, true, f, M, K, out));
    ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

template <int K>
static int launch_posterior(const ChunkLayout& lay, const double* Kuu, const double* acc, double sigma2,
                            double* alpha, double* S, double* info, char* work, cudaStream_t st) {
    PosteriorArgs<K> a;
    a.lay = lay;
    char* p = work;
    for (int c = 0; c < 2; ++c) { a.cols[c] = ChainPlan<double, K>::carve(lay, p); p += ChainPlan<double, K>::bytes(lay); }
    const int M = lay.M;
    const size_t band_bytes = (((size_t)(K + 1) * M * sizeof(double)) + 255) & ~(size_t)255;
    a.sigK = reinterpret_cast<double*>(p); p += band_bytes;
    a.sigP = reinterpret_cast<double*>(p); p += band_bytes;
    a.x = reinterpret_cast<double*>(p);
    p += ((size_t)M * sizeof(double) + 255) & ~(size_t)255;
    a.Kuu = Kuu; a.G = acc; a.b = acc + (size_t)(K + 1) * M;
    a.sigma2 = sigma2;
    a.info = info;
    {
        using T = double;
        T* rows = reinterpret_cast<T*>(p);
        a.rows = rows;
        ChainSpec<T> s0{BandMat<T>{Kuu, nullptr, nullptr, 0.0, 0.0, 0, M}, VecRhs<T>{Kuu, M, 0}};
        ChainSpec<T> s1{BandMat<T>{Kuu, nullptr, a.G, 1.0 / sigma2, 0.0, 0, M}, VecRhs<T>{a.b, M, 1}};
        const size_t total = 2 * chain_rows_count<T, K>(lay);
        chain_rows_kernel<T, K, 2><<<(int)std::min<size_t>((total + 255) / 256, 148 * 8), 256, 0, st>>>(lay, s0, s1, s1, s1, rows); ASVGP_LAUNCHED();
        ASVGP_CUDA_OK(cudaGetLastError());
    }
    ASVGP_CUDA_OK(cudaMemsetAsync(a.sigK, 0, 2 * band_bytes, st));
    const size_t smem = ChainSmall<double, K>::bytes(lay.P);
    ASVGP_CUDA_OK(cudaFuncSetAttribute(posterior_chains_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    posterior_chains_kernel<K><<<2, kChainThreads, smem, st>>>(a); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    const int band_elems = (K + 1) * M;
    posterior_combine_kernel<<<(band_elems + 255) / 256, 256, 0, st>>>(a.sigK, a.sigP, a.x, 1.0 / sigma2, M, band_elems,
                                                                      alpha, S); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

template <int K>
static int max_chunks_for_smem() {
    int P = kChainThreads;
    while (P > 1 && ChainSmall<Dual<1>, K>::bytes(P) > kChainSmemLimit) --P;
    return P;
}

static ChunkLayout pick_layout(int M, int K, int chunks) {
    int P = chunks > 0 ? chunks : default_chunks(M, K);
    int cap = kChainThreads;
    switch (K) {
        case 1: cap = max_chunks_for_smem<1>(); break;
        case 2: cap = max_chunks_for_smem<2>(); break;
        case 3: cap = max_chunks_for_smem<3>(); break;
        case 4: cap = max_chunks_for_smem<4>(); break;
        case 5: cap = max_chunks_for_smem<5>(); break;
        case 6: cap = max_chunks_for_smem<6>(); break;
    }
    if (P > cap) P = cap;
    return make_layout(M, K, P);
}

// Layout of the ELBO + gradient chains: with the library default (chunks = 0) and enough columns, 128 * n_cta chunks on a
// cluster of n_cta CTAs per chain (run_chain_cluster); n_cta = 8 (4, 2 when M is too small), ASVGP_CHAIN_CTAS overrides (1 = single CTA).
// chunks = 256 / 512 / 1024 asks for a cluster of 2 / 4 / 8 CTAs explicitly (the Kuu chain that runs beside the accumulate takes 4).
static ChunkLayout pick_layout_elbo(int M, int K, int chunks) {
    const bool explicit_cluster = chunks == 2 * kChainThreads || chunks == 4 * kChainThreads || chunks == 8 * kChainThreads;
    const ChunkLayout one = pick_layout(M, K, explicit_cluster ? 0 : chunks);
    if ((chunks != 0 && !explicit_cluster) || one.P < kChainThreads) return one;
    int n_cta = explicit_cluster ? chunks / kChainThreads : 8;
    if (const char* e = getenv("ASVGP_CHAIN_CTAS")) n_cta = atoi(e);
    if (n_cta != 2 && n_cta != 4 && n_cta != 8) return one;
    int P = M / (2 * (K + 1) + 1);                                 // chunk interiors of at least K + 1 columns with room to spare
    while (n_cta > 1 && P < kChainThreads * n_cta) n_cta /= 2;     // whole CTAs of 128 lanes only
    if (n_cta <= 1) return one;
    return make_layout(M, K, kChainThreads * n_cta);
}

}  // namespace asvgp

using namespace asvgp;

#define ASVGP_DISPATCH_ORDER(order, CALL)                         \
    switch (order) {                                              \
        case 1: { constexpr int K = 1; CALL; } break;             \
        case 2: { constexpr int K = 2; CALL; } break;             \
        case 3: { constexpr int K = 3; CALL; } break;             \
        case 4: { constexpr int K = 4; CALL; } break;             \
        case 5: { constexpr int K = 5; CALL; } break;             \
        case 6: { constexpr int K = 6; CALL; } break;             \
        default:                                                  \
            set_last_error("spline order %d not in 1..6", order); \
            return kBadArgument;                                  \
    }

extern "C" int asvgp_kuu_assemble(const double* tables, int n_terms, const double* h_coef, const double* h_dcoef,
                                  int M, int order, double* Kuu, double* dKuu, void* stream) {
    ASVGP_REQUIRE(n_terms >= 1 && n_terms <= kMaxTerms, "kuu_assemble: n_terms=%d not in 1..%d", n_terms, kMaxTerms);
    ASVGP_REQUIRE(M > 0 && order >= 1 && order <= kMaxOrder, "kuu_assemble: M=%d order=%d", M, order);
    KuuTerms t;
    t.n_terms = n_terms;
    for (int i = 0; i < n_terms; ++i) { t.coef[i] = h_coef[i]; t.dcoef[i] = h_dcoef ? h_dcoef[i] : 0.0; }
    const int64_t elems = (int64_t)(order + 1) * M;
    const int blocks = (int)((elems + 255) / 256);
    kuu_assemble_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(tables, t, elems, Kuu, dKuu); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

extern "C" int asvgp_kuu_assemble_batched(const double* tables, int n_terms, int B, const double* h_coef, const double* h_dcoef,
                                          int M, int order, double* Kuu, double* dKuu, void* stream) {
    ASVGP_REQUIRE(n_terms >= 1 && n_terms <= kMaxTerms, "kuu_assemble_batched: n_terms=%d not in 1..%d", n_terms, kMaxTerms);
    ASVGP_REQUIRE(B >= 1 && B <= ASVGP_MAX_BATCH, "kuu_assemble_batched: B=%d not in 1..%d", B, ASVGP_MAX_BATCH);
    ASVGP_REQUIRE(M > 0 && order >= 1 && order <= kMaxOrder, "kuu_assemble_batched: M=%d order=%d", M, order);
    ASVGP_REQUIRE(h_coef != nullptr, "kuu_assemble_batched: h_coef is NULL");
    KuuTermsBatch t;
    t.n_terms = n_terms;
    for (int b = 0; b < B; ++b)
        for (int i = 0; i < n_terms; ++i) {
            t.coef[b][i] = h_coef[b * n_terms + i];
            t.dcoef[b][i] = h_dcoef ? h_dcoef[b * n_terms + i] : 0.0;
        }
    const int64_t elems = (int64_t)(order + 1) * M;
    const dim3 grid((unsigned)((elems + 255) / 256), B);
    kuu_assemble_batched_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(tables, t, elems, Kuu, dKuu); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

// Every layout pick_layout_elbo may choose for (M, order, chunks) (ASVGP_CHAIN_CTAS can change it between calls); cand[0] is
// the single-CTA layout of pick_layout.
static int elbo_layout_candidates(int M, int order, int chunks, ChunkLayout cand[4]) {
    const ChunkLayout lay = pick_layout(M, order, chunks > kChainThreads ? 0 : chunks);
    int n_cand = 0;
    cand[n_cand++] = lay;
    if ((chunks == 0 || chunks == 2 * kChainThreads || chunks == 4 * kChainThreads || chunks == 8 * kChainThreads) && lay.P >= kChainThreads) {
        const int P = M / (2 * (order + 1) + 1);
        if (P >= 2 * kChainThreads) cand[n_cand++] = make_layout(M, order, 2 * kChainThreads);
        if (P >= 4 * kChainThreads) cand[n_cand++] = make_layout(M, order, 4 * kChainThreads);
        if (P >= 8 * kChainThreads) cand[n_cand++] = make_layout(M, order, 8 * kChainThreads);
    }
    return n_cand;
}

extern "C" int64_t asvgp_workspace_bytes_1d(int M, int order, int chunks) {
    if (M <= 0 || order < 1 || order > kMaxOrder) return -1;
    // the ELBO chains may run on a clustered layout (pick_layout_elbo; ASVGP_CHAIN_CTAS): size for every candidate
    ChunkLayout cand[4];
    const int n_cand = elbo_layout_candidates(M, order, chunks, cand);
    const ChunkLayout lay = cand[0];
    size_t e = 0, p = 0;
    for (int c = 0; c < n_cand; ++c) {
        size_t ec = 0;
        switch (order) {
            case 1: ec = elbo_work_bytes<1>(cand[c]); p = posterior_work_bytes<1>(lay); break;
            case 2: ec = elbo_work_bytes<2>(cand[c]); p = posterior_work_bytes<2>(lay); break;
            case 3: ec = elbo_work_bytes<3>(cand[c]); p = posterior_work_bytes<3>(lay); break;
            case 4: ec = elbo_work_bytes<4>(cand[c]); p = posterior_work_bytes<4>(lay); break;
            case 5: ec = elbo_work_bytes<5>(cand[c]); p = posterior_work_bytes<5>(lay); break;
            case 6: ec = elbo_work_bytes<6>(cand[c]); p = posterior_work_bytes<6>(lay); break;
        }
        e = ec > e ? ec : e;
    }
    return (int64_t)(e > p ? e : p);
}

extern "C" int64_t asvgp_workspace_bytes_1d_batched(int M, int order, int chunks, int B, int D) {
    if (M <= 0 || order < 1 || order > kMaxOrder || B < 1 || B > ASVGP_MAX_BATCH || D < 1 || D > ASVGP_MAX_BATCH_COLUMNS) return -1;
    ChunkLayout cand[4];
    const int n_cand = elbo_layout_candidates(M, order, chunks, cand);
    size_t e = 0;
    for (int c = 0; c < n_cand; ++c) {
        size_t ec = 0;
        switch (order) {
            case 1: ec = BatchPlan<1>(cand[c], B, D).total; break;
            case 2: ec = BatchPlan<2>(cand[c], B, D).total; break;
            case 3: ec = BatchPlan<3>(cand[c], B, D).total; break;
            case 4: ec = BatchPlan<4>(cand[c], B, D).total; break;
            case 5: ec = BatchPlan<5>(cand[c], B, D).total; break;
            case 6: ec = BatchPlan<6>(cand[c], B, D).total; break;
        }
        e = ec > e ? ec : e;
    }
    return (int64_t)e;
}

extern "C" int asvgp_elbo_grad_1d(const double* Kuu, const double* dKuu, const double* acc, int M, int order,
                                  double variance, double sigma2, int chunks, double* out, void* work,
                                  int64_t work_bytes, void* stream) {
    ASVGP_REQUIRE(M > 2 * order && order >= 1 && order <= kMaxOrder, "elbo_grad_1d: M=%d order=%d", M, order);
    ASVGP_REQUIRE(variance > 0.0 && sigma2 > 0.0, "elbo_grad_1d: variance=%g sigma2=%g must be positive", variance, sigma2);
    ASVGP_REQUIRE(work_bytes >= asvgp_workspace_bytes_1d(M, order, chunks), "elbo_grad_1d: workspace too small");
    const ChunkLayout lay = pick_layout_elbo(M, order, chunks);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ASVGP_DISPATCH_ORDER(order, { if (int rc = launch_elbo<K>(lay, Kuu, dKuu, acc, variance, sigma2, out,
                                                              static_cast<char*>(work), st)) return rc; });
    return kOk;
}

extern "C" int asvgp_elbo_grad_1d_batched(const double* Kuu, const double* dKuu, const double* acc, int M, int order, int B, int D,
                                          const double* h_variance, const double* h_sigma2, int chunks, double* out, void* work,
                                          int64_t work_bytes, void* stream) {
    ASVGP_REQUIRE(M > 2 * order && order >= 1 && order <= kMaxOrder, "elbo_grad_1d_batched: M=%d order=%d", M, order);
    ASVGP_REQUIRE(B >= 1 && B <= ASVGP_MAX_BATCH, "elbo_grad_1d_batched: B=%d not in 1..%d", B, ASVGP_MAX_BATCH);
    ASVGP_REQUIRE(D >= 1 && D <= ASVGP_MAX_BATCH_COLUMNS, "elbo_grad_1d_batched: D=%d not in 1..%d", D, ASVGP_MAX_BATCH_COLUMNS);
    ASVGP_REQUIRE(h_variance != nullptr && h_sigma2 != nullptr, "elbo_grad_1d_batched: h_variance / h_sigma2 is NULL");
    for (int b = 0; b < B; ++b)
        ASVGP_REQUIRE(h_variance[b] > 0.0 && h_sigma2[b] > 0.0, "elbo_grad_1d_batched: slot %d: variance=%g sigma2=%g must be positive",
                      b, h_variance[b], h_sigma2[b]);
    ASVGP_REQUIRE(work_bytes >= asvgp_workspace_bytes_1d_batched(M, order, chunks, B, D), "elbo_grad_1d_batched: workspace too small");
    const ChunkLayout lay = pick_layout_elbo(M, order, chunks);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ASVGP_DISPATCH_ORDER(order, { if (int rc = launch_elbo_batched<K>(lay, B, D, Kuu, dKuu, acc, h_variance, h_sigma2, out,
                                                                      static_cast<char*>(work), st)) return rc; });
    return kOk;
}

extern "C" int64_t asvgp_kuu_state_doubles(int M, int order) {
    if (M <= 0 || order < 1 || order > kMaxOrder) return -1;
    return (int64_t)kuu_state_doubles(M, order);
}

extern "C" int asvgp_kuu_chain_1d(const double* Kuu, const double* dKuu, int M, int order, int chunks, double* kuu_state,
                                  void* work, int64_t work_bytes, void* gate_event, void* stream) {
    ASVGP_REQUIRE(M > 2 * order && order >= 1 && order <= kMaxOrder, "kuu_chain_1d: M=%d order=%d", M, order);
    ASVGP_REQUIRE(work_bytes >= asvgp_workspace_bytes_1d(M, order, chunks), "kuu_chain_1d: workspace too small");
    const ChunkLayout lay = pick_layout_elbo(M, order, chunks);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ASVGP_DISPATCH_ORDER(order, { if (int rc = launch_kuu_chain<K>(lay, Kuu, dKuu, kuu_state, static_cast<char*>(work),
                                                                   static_cast<cudaEvent_t>(gate_event), st)) return rc; });
    return kOk;
}

extern "C" int asvgp_elbo_grad_1d_prepared(const double* kuu_state, const double* Kuu, const double* dKuu, const double* acc,
                                           int M, int order, double variance, double sigma2, int chunks, double* out,
                                           void* work, int64_t work_bytes, void* kuu_ready_event, int join_late, void* stream) {
    ASVGP_REQUIRE(M > 2 * order && order >= 1 && order <= kMaxOrder, "elbo_grad_1d_prepared: M=%d order=%d", M, order);
    ASVGP_REQUIRE(variance > 0.0 && sigma2 > 0.0, "elbo_grad_1d_prepared: variance=%g sigma2=%g must be positive", variance, sigma2);
    ASVGP_REQUIRE(work_bytes >= asvgp_workspace_bytes_1d(M, order, chunks), "elbo_grad_1d_prepared: workspace too small");
    const ChunkLayout lay = pick_layout_elbo(M, order, chunks);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ASVGP_DISPATCH_ORDER(order, { if (int rc = launch_pchains<K>(lay, kuu_state, Kuu, dKuu, acc, variance, sigma2, out, static_cast<char*>(work),
                                                                 static_cast<cudaEvent_t>(kuu_ready_event), join_late, st)) return rc; });
    return kOk;
}

extern "C" int asvgp_posterior_1d(const double* Kuu, const double* acc, int M, int order, double sigma2, int chunks,
                                  double* alpha, double* S_band, double* info, void* work, int64_t work_bytes,
                                  void* stream) {
    ASVGP_REQUIRE(M > 2 * order && order >= 1 && order <= kMaxOrder, "posterior_1d: M=%d order=%d", M, order);
    ASVGP_REQUIRE(sigma2 > 0.0, "posterior_1d: sigma2=%g must be positive", sigma2);
    ASVGP_REQUIRE(work_bytes >= asvgp_workspace_bytes_1d(M, order, chunks), "posterior_1d: workspace too small");
    const ChunkLayout lay = pick_layout(M, order, chunks);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ASVGP_DISPATCH_ORDER(order, { if (int rc = launch_posterior<K>(lay, Kuu, acc, sigma2, alpha, S_band, info,
                                                                   static_cast<char*>(work), st)) return rc; });
    return kOk;
}

extern "C" int asvgp_band_inverse_1d(const double* A, const double* dA, int M, int order, int chunks, double* sig_val,
                                     double* sig_tan, double* scal, void* work, int64_t work_bytes, void* stream) {
    ASVGP_REQUIRE(M > 2 * order && order >= 1 && order <= kMaxOrder, "band_inverse_1d: M=%d order=%d", M, order);
    ASVGP_REQUIRE(work_bytes >= asvgp_workspace_bytes_1d(M, order, chunks), "band_inverse_1d: workspace too small");
    const ChunkLayout lay = pick_layout(M, order, chunks);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ASVGP_DISPATCH_ORDER(order, { if (int rc = launch_band_inverse<K>(lay, A, dA, sig_val, sig_tan, scal,
                                                                      static_cast<char*>(work), st)) return rc; });
    return kOk;
}
