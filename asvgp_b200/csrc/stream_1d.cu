// Streaming (HBM-bound) 1-D kernels: Kuf evaluation, fused Gram/projection accumulation, posterior predictor.
//
//   asvgp_basis_eval_1d  <- SplineBasis.evaluate_basis        (reference asvgp/basis.py:51-80)
//   asvgp_accum_1d       <- GPR_1d.__init__ precompute        (reference asvgp/gpr.py:39-44, utils.py:24-30)
//   asvgp_predict_1d     <- GPR_1d.predict_f                  (reference asvgp/gpr.py:91-136)
//
// accum_1d design (DESIGN.md §4.1).  Kuf is never materialised.  Each CTA streams one contiguous slice of (x, y)
// with 128-bit read-only loads, U=4 loads of x and of y in flight per thread.  Every warp keeps, in registers, the
// (k+1)(k+2)/2 + (k+1) partial sums of w w^T and w*y for ONE knot interval `cur` (warp-uniform).  While the
// points a warp reads stay inside that interval (time-series / raster order: ~N/M consecutive points do) the inner
// loop is pure register FMAs.  When a warp meets a point of another interval it butterfly-reduces its partial sums
// with warp shuffles and issues one fp64 RED per band entry, then switches interval.  Points that belong to neither
// the old nor the new interval (only possible for unsorted input) are added with per-point REDs, so any input order
// gives the right answer; sorted input costs ~(k+1)(k+4)/2 REDs per warp per interval crossing, i.e. nothing.
// x and y may each be float32 or float64 (asvgp_accum_1d_typed): they are loaded in their own type and converted to double in
// registers, so a float32 pair streams 8 B per point instead of 16 through the same fp64 arithmetic.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>

#include "common.cuh"
#include "partition.cuh"
#include "../../include/asvgp_b200.h"

namespace asvgp {

// x0 and delta = mesh[1]-mesh[0] (reference basis.py:18) are read from the device-resident mesh by the kernel
// itself, so no entry point has to synchronise with the host to learn them.
__device__ __forceinline__ Mesh load_mesh(const double* knots, int n_knots) {
    Mesh m;
    m.knots = knots;
    m.n_knots = n_knots;
    m.x0 = __ldg(knots);
    m.inv_delta = 1.0 / (__ldg(knots + 1) - m.x0);
    return m;
}

__device__ __forceinline__ int64_t imin64(int64_t a, int64_t b) { return a < b ? a : b; }

struct LdgLoader {
    __device__ __forceinline__ double operator()(const double* p) const { return __ldg(p); }
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ------------------------------------------------------------------------------------------------------------------
// basis evaluation (API parity with evaluate_basis; materialises the (k+1) n non-zeros)
// ------------------------------------------------------------------------------------------------------------------
template <int K>
__global__ void __launch_bounds__(256) basis_eval_1d_kernel(const double* __restrict__ x, int64_t n, const double* __restrict__ knots, int n_knots,
                                                            int dx, const double* __restrict__ coef,
                                                            int64_t* __restrict__ idx_out,
                                                            double* __restrict__ vals) {
    __shared__ double s_coef[(K + 1) * (K + 1)];
    if (dx > 0) {
        for (int i = threadIdx.x; i < (K + 1) * (K + 1); i += blockDim.x) s_coef[i] = coef[i];
        __syncthreads();
    }
    const Mesh mesh = load_mesh(knots, n_knots);
    double scale = 1.0;
    for (int i = 0; i < dx; ++i) scale *= mesh.inv_delta;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double xi = x[i];
        const int idx = locate_interval(mesh, xi, LdgLoader());
        const double t = (xi - __ldg(mesh.knots + idx)) * mesh.inv_delta;
        double w[K + 1];
        if (dx == 0) bspline_pieces<K>(t, w);
        else bspline_pieces_coef<K>(t, s_coef, scale, w);
        idx_out[i] = idx;
#pragma unroll
        for (int r = 0; r <= K; ++r) vals[(int64_t)r * n + i] = w[r];
    }
}

// ------------------------------------------------------------------------------------------------------------------
// fused accumulation
// ------------------------------------------------------------------------------------------------------------------
constexpr int kAccumThreads = 256;
constexpr int kAccumUnroll = 8;

template <int K>
struct WarpAccum {
    static constexpr int kPairs = Counts<K>::kPairs;
    static constexpr int kAcc = Counts<K>::kAcc;
    static constexpr int NG = 2 * K;          // Gram moments sum tau^j, j = 1..2K (j = 0 is the point count)
    static constexpr int NY = K + 1;          // projection moments sum y tau^j, j = 0..K
    double mg[NG], my[NY];
    int cnt;          // points added by this lane
    int cur;          // interval the register sums belong to (warp-uniform), -1 = none
    double u;         // mesh[cur]
    double lo, hi;    // x in (lo, hi]  <=>  locate_interval(x) == cur
    bool dirty;       // warp-uniform: the sums hold something

    __device__ __forceinline__ void clear() {
#pragma unroll
        for (int i = 0; i < NG; ++i) mg[i] = 0.0;
#pragma unroll
        for (int i = 0; i < NY; ++i) my[i] = 0.0;
        cnt = 0;
        dirty = false;
    }
    __device__ __forceinline__ void set_interval(const Mesh& mesh, int idx) {
        cur = idx;
        u = __ldg(mesh.knots + idx);
        lo = (idx == 0) ? -INFINITY : u;
        hi = (idx == mesh.n_knots - 2) ? INFINITY : __ldg(mesh.knots + idx + 1);
    }
    __device__ __forceinline__ bool inside(double x) const { return x > lo && x <= hi; }

    // centred monomial moments of the point (see MomentCoef in common.cuh): 5K+2 fp64 instructions
    __device__ __forceinline__ void add(const Mesh& mesh, double x, double y) {
        add_tau(fma(x - u, mesh.inv_delta, -0.5), y);
    }
    __device__ __forceinline__ void add_tau(double tau, double y) {
        double p = tau;
        mg[0] += p;
        my[0] += y;
#pragma unroll
        for (int j = 2; j <= NG; ++j) {
            if (j - 1 <= K) my[j - 1] = fma(y, p, my[j - 1]);        // y tau^(j-1)
            p *= tau;
            mg[j - 1] += p;
        }
        ++cnt;
    }
    // shuffle-reduce the moments over the warp, convert them to band entries and add those to the band: one RED per
    // entry per warp, issued by lane `entry`
    __device__ __forceinline__ void flush(double* __restrict__ G, double* __restrict__ b, int M, int lane) {
        if (dirty) {
            double Mg[NG + 1], My[NY];
            Mg[0] = (double)__reduce_add_sync(0xffffffffu, cnt);
#pragma unroll
            for (int j = 0; j < NG; ++j) Mg[j + 1] = warp_sum(mg[j]);
#pragma unroll
            for (int j = 0; j < NY; ++j) My[j] = warp_sum(my[j]);
            const MomentCoef<K>& mc = g_moment_coef<K>;
#pragma unroll
            for (int e0 = 0; e0 < kAcc; e0 += 32) {               // kAcc = 35 for K = 6: a second round for three entries
                const int e = e0 + lane;
                if (e < kPairs) {
                    double v = 0.0;
#pragma unroll
                    for (int j = 0; j <= NG; ++j) v = fma(mc.cg[e][j], Mg[j], v);
                    const int r = mc.rr[e], s = mc.ss[e];
                    atomicAdd(G + (int64_t)(r - s) * M + cur + s, v);
                } else if (e < kAcc) {
                    const int r = e - kPairs;
                    double v = 0.0;
#pragma unroll
                    for (int j = 0; j < NY; ++j) v = fma(mc.cb[r][j], My[j], v);
                    atomicAdd(b + cur + r, v);
                }
            }
        }
        clear();
    }
};

// Same as WarpAccum::flush for GL-lane groups that each hold their own interval: the moments are reduced inside every
// group (log2 GL shuffle steps serve all 32/GL groups at once), lane l of a group converts and adds entries l, l + GL, ...
template <int K, int GL>
__device__ __forceinline__ void flush_groups(WarpAccum<K>& wa, bool any, double* __restrict__ G, double* __restrict__ b, int M, int lane) {
    constexpr int NG = WarpAccum<K>::NG, NY = WarpAccum<K>::NY, kPairs = WarpAccum<K>::kPairs, kAcc = WarpAccum<K>::kAcc;
    double Mg[NG + 1], My[NY];
    int c = wa.cnt;
#pragma unroll
    for (int o = GL / 2; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    Mg[0] = (double)c;
#pragma unroll
    for (int j = 0; j < NG; ++j) {
        double v = wa.mg[j];
#pragma unroll
        for (int o = GL / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        Mg[j + 1] = v;
    }
#pragma unroll
    for (int j = 0; j < NY; ++j) {
        double v = wa.my[j];
#pragma unroll
        for (int o = GL / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        My[j] = v;
    }
    if (any) {
        const MomentCoef<K>& mc = g_moment_coef<K>;
#pragma unroll
        for (int e0 = 0; e0 < kAcc; e0 += GL) {
            const int e = e0 + (lane & (GL - 1));
            if (e < kPairs) {
                double v = 0.0;
#pragma unroll
                for (int j = 0; j <= NG; ++j) v = fma(mc.cg[e][j], Mg[j], v);
                const int r = mc.rr[e], q = mc.ss[e];
                atomicAdd(G + (int64_t)(r - q) * M + wa.cur + q, v);
            } else if (e < kAcc) {
                const int r = e - kPairs;
                double v = 0.0;
#pragma unroll
                for (int j = 0; j < NY; ++j) v = fma(mc.cb[r][j], My[j], v);
                atomicAdd(b + wa.cur + r, v);
            }
        }
    }
    wa.clear();
}

// one point straight to global memory (unsorted-input slow path)
template <int K>
__device__ __forceinline__ void scatter_point(const Mesh& mesh, int idx, double x, double y,
                                              double* __restrict__ G, double* __restrict__ b, int M) {
    const double t = (x - __ldg(mesh.knots + idx)) * mesh.inv_delta;
    double w[K + 1];
    bspline_pieces<K>(t, w);
#pragma unroll
    for (int r = 0; r <= K; ++r) {
#pragma unroll
        for (int s = 0; s <= r; ++s) atomicAdd(G + (int64_t)(r - s) * M + idx + s, w[r] * w[s]);
        atomicAdd(b + idx + r, w[r] * y);
    }
}

// VEC consecutive points of one array from a 16-byte aligned address, evict-first: double2 loads, or one float4
template <int VEC>
__device__ __forceinline__ void ldg_stream_vec(const double* p, double (&v)[VEC], uint64_t pol) {
#pragma unroll
    for (int h = 0; h < VEC; h += 2) {
        const double2 d = ldg_stream2(p + h, pol);
        v[h] = d.x; v[h + 1] = d.y;
    }
}
template <int VEC>
__device__ __forceinline__ void ldg_stream_vec(const float* p, float (&v)[VEC], uint64_t pol) {
    static_assert(VEC == 4, "float32 points are read four at a time");
    const float4 f = ldg_stream4f(p, pol);
    v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
}

// Slots in flight per lane.  2-point float64 slots: 8 (256 B).  4-point slots carry four copies of the per-point code, so
// fewer of them fit the 128 registers of two CTAs per SM without spilling at k = 3: 6 for a float32 pair (24 points,
// 192 B), 4 for a mixed pair (16 points, 192 B).
template <int VEC, class TX, class TY>
constexpr int accum_unroll() { return VEC == 4 ? (sizeof(TX) == sizeof(TY) ? 6 : 4) : kAccumUnroll; }

// The U slots of one warp tile: VEC points per slot from 16-byte aligned addresses (VEC > 1) or scalar loads (VEC = 1).
template <int U, int VEC, class TX, class TY>
__device__ __forceinline__ void load_tile(const TX* __restrict__ x, const TY* __restrict__ y, int64_t n, int64_t slot0,
                                          TX (&xs)[U][VEC], TY (&ys)[U][VEC], uint64_t stream_policy) {
#pragma unroll
    for (int j = 0; j < U; ++j) {
        const int64_t slot = slot0 + j * 32;
        const int64_t p = slot * VEC;
        if constexpr (VEC > 1) {
            if (p + VEC - 1 < n) {
                ldg_stream_vec<VEC>(x + p, xs[j], stream_policy);
                ldg_stream_vec<VEC>(y + p, ys[j], stream_policy);
            } else {
                // the array's tail: entries past n (never added) repeat the slot's first x
#pragma unroll
                for (int e = 0; e < VEC; ++e) {
                    xs[j][e] = (p + e < n) ? __ldg(x + p + e) : (e ? xs[j][0] : (TX)0);
                    ys[j][e] = (p + e < n) ? __ldg(y + p + e) : (TY)0;
                }
            }
        } else {
            xs[j][0] = (p < n) ? __ldg(x + p) : (TX)0;
            ys[j][0] = (p < n) ? __ldg(y + p) : (TY)0;
        }
    }
}

// One slot whose points do not all lie in the warp's interval: the points of `valid` inside it join the register sums, which are
// flushed; the warp adopts the interval of the highest lane's outside point (at least one lane must have one), and outside
// points of any other interval go to global memory one by one.
template <int K, int VEC>
__device__ __forceinline__ void cross_interval(WarpAccum<K>& wa, const Mesh& mesh, const double (&xd)[VEC], const double (&yd)[VEC],
                                               const bool (&valid)[VEC], const bool (&in)[VEC], double* __restrict__ G,
                                               double* __restrict__ b, int M, int lane) {
    int where[VEC];
    bool pending = false, added_old = false;
    int cand = -1;
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
        where[e] = -1;
        if (valid[e]) {
            if (in[e]) { wa.add(mesh, xd[e], yd[e]); added_old = true; }
            else {
                where[e] = locate_interval(mesh, xd[e], LdgLoader());
                pending = true;
                cand = where[e];
            }
        }
    }
    // (cur == -1 before the first point: nothing accumulated yet, nothing to flush)
    wa.dirty = wa.dirty || __any_sync(0xffffffffu, added_old);
    wa.flush(G, b, M, lane);
    const unsigned pend = __ballot_sync(0xffffffffu, pending);   // non-zero here
    const int src = 31 - __clz(pend);
    wa.set_interval(mesh, __shfl_sync(0xffffffffu, cand, src));
    bool added = false;
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
        if (where[e] >= 0) {
            if (where[e] == wa.cur) { wa.add(mesh, xd[e], yd[e]); added = true; }
            else scatter_point<K>(mesh, where[e], xd[e], yd[e], G, b, M);
        }
    }
    wa.dirty = __any_sync(0xffffffffu, added);
}

// x and y hold float64 or float32 (TX, TY); the values stay in their own type until they are used and are converted to
// double there (exact).  VEC = 2: both arrays are float64 and 16-byte aligned and are read as double2; VEC = 4: at least
// one is float32, both are 16-byte aligned, a slot is 4 points (float4, or 2 x double2); VEC = 1: scalar loads
// (misaligned views).
template <int K, int VEC, class TX, class TY>
__global__ void __launch_bounds__(kAccumThreads, 2)
accum_1d_kernel(const TX* __restrict__ x, const TY* __restrict__ y, int64_t n,
                const double* __restrict__ knots, int n_knots, int M,
                double* __restrict__ G, double* __restrict__ b, double* __restrict__ scal) {
    constexpr int U = accum_unroll<VEC, TX, TY>();
    const Mesh mesh = load_mesh(knots, n_knots);
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    constexpr int kWarps = kAccumThreads / 32;

    // slots of VEC points; CTA c owns a contiguous range of whole warp-tiles (32*U slots)
    const int64_t n_slots = (n + VEC - 1) / VEC;
    const int64_t tile = 32 * U;
    const int64_t n_tiles = (n_slots + tile - 1) / tile;
    const int64_t tiles_per_cta = (n_tiles + gridDim.x - 1) / gridDim.x;
    const int64_t t_begin = blockIdx.x * tiles_per_cta;
    const int64_t t_end = imin64(t_begin + tiles_per_cta, n_tiles);

    WarpAccum<K> wa;
    wa.clear();
    wa.cur = -1;
    wa.u = 0.0;
    wa.lo = INFINITY;
    wa.hi = -INFINITY;
    double yy = 0.0;
    const uint64_t stream_policy = evict_first_policy();

    // within the CTA's range warp w takes the w-th contiguous share, so that (for ordered input) each warp meets as
    // few interval crossings as possible
    const int64_t my_tiles = t_end > t_begin ? t_end - t_begin : 0;
    const int64_t per_warp = (my_tiles + kWarps - 1) / kWarps;
    const int64_t w_begin = t_begin + warp * per_warp;
    const int64_t w_end = imin64(w_begin + per_warp, t_end);

    for (int64_t tl = w_begin; tl < w_end; ++tl) {
        TX xs[U][VEC];
        TY ys[U][VEC];
        const int64_t slot0 = tl * tile + lane;
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int64_t slot = slot0 + j * 32;
            const int64_t p = slot * VEC;
            if constexpr (VEC > 1) {
                if (p + VEC - 1 < n) {
                    ldg_stream_vec<VEC>(x + p, xs[j], stream_policy);
                    ldg_stream_vec<VEC>(y + p, ys[j], stream_policy);
                } else {
                    // the array's tail: entries past n (never added) repeat the slot's first x
#pragma unroll
                    for (int e = 0; e < VEC; ++e) {
                        xs[j][e] = (p + e < n) ? __ldg(x + p + e) : (e ? xs[j][0] : (TX)0);
                        ys[j][e] = (p + e < n) ? __ldg(y + p + e) : (TY)0;
                    }
                }
            } else {
                xs[j][0] = (p < n) ? __ldg(x + p) : (TX)0;
                ys[j][0] = (p < n) ? __ldg(y + p) : (TY)0;
            }
        }
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int64_t p = (slot0 + j * 32) * VEC;
            double xd[VEC], yd[VEC];
#pragma unroll
            for (int e = 0; e < VEC; ++e) { xd[e] = (double)xs[j][e]; yd[e] = (double)ys[j][e]; }
            bool valid[VEC], in[VEC];
            bool all_in = true;
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                valid[e] = (p + e) < n;
                in[e] = wa.inside(xd[e]);
                all_in = all_in && (in[e] || !valid[e]);
                if (valid[e]) yy = fma(yd[e], yd[e], yy);
            }
            if (__all_sync(0xffffffffu, all_in)) {
#pragma unroll
                for (int e = 0; e < VEC; ++e)
                    if (valid[e]) wa.add(mesh, xd[e], yd[e]);
                wa.dirty = true;
            } else {
                // interval crossing (or unsorted input)
                int where[VEC];
                bool pending = false, added_old = false;
                int cand = -1;
#pragma unroll
                for (int e = 0; e < VEC; ++e) {
                    where[e] = -1;
                    if (valid[e]) {
                        if (in[e]) { wa.add(mesh, xd[e], yd[e]); added_old = true; }
                        else {
                            where[e] = locate_interval(mesh, xd[e], LdgLoader());
                            pending = true;
                            cand = where[e];
                        }
                    }
                }
                // (cur == -1 before the first point: nothing accumulated yet, nothing to flush)
                wa.dirty = wa.dirty || __any_sync(0xffffffffu, added_old);
                wa.flush(G, b, M, lane);
                const unsigned pend = __ballot_sync(0xffffffffu, pending);   // non-zero here
                const int src = 31 - __clz(pend);
                wa.set_interval(mesh, __shfl_sync(0xffffffffu, cand, src));
                bool added = false;
#pragma unroll
                for (int e = 0; e < VEC; ++e) {
                    if (where[e] >= 0) {
                        if (where[e] == wa.cur) { wa.add(mesh, xd[e], yd[e]); added = true; }
                        else scatter_point<K>(mesh, where[e], xd[e], yd[e], G, b, M);
                    }
                }
                wa.dirty = __any_sync(0xffffffffu, added);
            }
        }
    }
    wa.flush(G, b, M, lane);

    __shared__ double s_yy[kWarps];
    yy = warp_sum(yy);
    if (lane == 0) s_yy[warp] = yy;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) tot += s_yy[w];
        atomicAdd(scal, tot);
        if (blockIdx.x == 0) atomicAdd(scal + 1, (double)n);
    }
}

// Series of point p (0 <= p < offsets[S]): the largest s with offsets[s] <= p, which skips empty series.
__device__ __forceinline__ int find_series(const int64_t* __restrict__ offsets, int S, int64_t p) {
    int lo = 0, hi = S - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(offsets + mid) <= p) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// S independent series concatenated in (x, y), series s being points offsets[s] .. offsets[s+1] - 1: accum_1d_kernel's tiles and
// register sums, with one packed accumulator per series (acc + s * ((K+2) M + 2)).  A warp tracks the series of its points
// (binary search for its first point, the series' end in a register).  A tile that lies inside the series runs accum_1d_kernel's
// slots after one warp-uniform compare.  A tile in which the series ends is walked slot by slot: a slot that crosses the end
// flushes the sums and sum(y^2) into that series, moves on to the series of the slot's last point and starts a new interval there;
// the points of series that lie wholly inside the slot go to their own accumulators one by one.
template <int K, int VEC, class TX, class TY>
__global__ void __launch_bounds__(kAccumThreads, 2)
accum_1d_segmented_kernel(const TX* __restrict__ x, const TY* __restrict__ y, int64_t n, const int64_t* __restrict__ offsets, int S,
                          const double* __restrict__ knots, int n_knots, int M, double* __restrict__ acc) {
    constexpr int U = accum_unroll<VEC, TX, TY>();
    const Mesh mesh = load_mesh(knots, n_knots);
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    constexpr int kWarps = kAccumThreads / 32;
    const int64_t L = (int64_t)(K + 2) * M + 2;

    const int64_t n_slots = (n + VEC - 1) / VEC;
    const int64_t tile = 32 * U;
    const int64_t n_tiles = (n_slots + tile - 1) / tile;
    const int64_t tiles_per_cta = (n_tiles + gridDim.x - 1) / gridDim.x;
    const int64_t t_begin = blockIdx.x * tiles_per_cta;
    const int64_t t_end = imin64(t_begin + tiles_per_cta, n_tiles);
    const int64_t my_tiles = t_end > t_begin ? t_end - t_begin : 0;
    const int64_t per_warp = (my_tiles + kWarps - 1) / kWarps;
    const int64_t w_begin = t_begin + warp * per_warp;
    const int64_t w_end = imin64(w_begin + per_warp, t_end);

    WarpAccum<K> wa;
    wa.clear();
    wa.cur = -1;
    wa.u = 0.0;
    wa.lo = INFINITY;
    wa.hi = -INFINITY;
    double yy = 0.0;
    const uint64_t stream_policy = evict_first_policy();

    int seg = -1;
    int64_t seg_end = 0;
    double* G = acc;
    if (w_begin < w_end) {
        seg = find_series(offsets, S, w_begin * tile * VEC);
        seg_end = __ldg(offsets + seg + 1);
        G = acc + seg * L;
    }

    for (int64_t tl = w_begin; tl < w_end; ++tl) {
        TX xs[U][VEC];
        TY ys[U][VEC];
        const int64_t slot0 = tl * tile + lane;
        load_tile<U, VEC>(x, y, n, slot0, xs, ys, stream_policy);
        if (imin64((tl + 1) * tile * VEC, n) <= seg_end) {
            // the tile lies inside the warp's series: accum_1d_kernel's slots
#pragma unroll
            for (int j = 0; j < U; ++j) {
                const int64_t p = (slot0 + j * 32) * VEC;
                double xd[VEC], yd[VEC];
#pragma unroll
                for (int e = 0; e < VEC; ++e) { xd[e] = (double)xs[j][e]; yd[e] = (double)ys[j][e]; }
                bool valid[VEC], in[VEC];
                bool all_in = true;
#pragma unroll
                for (int e = 0; e < VEC; ++e) {
                    valid[e] = (p + e) < n;
                    in[e] = wa.inside(xd[e]);
                    all_in = all_in && (in[e] || !valid[e]);
                    if (valid[e]) yy = fma(yd[e], yd[e], yy);
                }
                if (__all_sync(0xffffffffu, all_in)) {
#pragma unroll
                    for (int e = 0; e < VEC; ++e)
                        if (valid[e]) wa.add(mesh, xd[e], yd[e]);
                    wa.dirty = true;
                } else {
                    cross_interval<K, VEC>(wa, mesh, xd, yd, valid, in, G, G + (K + 1) * M, M, lane);
                }
            }
            continue;
        }
        // a series ends inside the tile: slot by slot, not unrolled (one copy of this code), the points read again (cached)
#pragma unroll 1
        for (int j = 0; j < U; ++j) {
            const int64_t p = (slot0 + j * 32) * VEC;
            const int64_t slot_last = imin64((tl * tile + j * 32 + 32) * VEC, n) - 1;      // warp-uniform
            double xd[VEC], yd[VEC];
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                xd[e] = (p + e < n) ? (double)__ldg(x + p + e) : 0.0;
                yd[e] = (p + e < n) ? (double)__ldg(y + p + e) : 0.0;
            }
            bool valid[VEC], in[VEC];
            bool all_in = true;
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                valid[e] = (p + e) < seg_end;
                in[e] = wa.inside(xd[e]);
                all_in = all_in && (in[e] || !valid[e]);
                if (valid[e]) yy = fma(yd[e], yd[e], yy);
            }
            if (slot_last < seg_end) {
                if (__all_sync(0xffffffffu, all_in)) {
#pragma unroll
                    for (int e = 0; e < VEC; ++e)
                        if (valid[e]) wa.add(mesh, xd[e], yd[e]);
                    wa.dirty = true;
                } else {
                    cross_interval<K, VEC>(wa, mesh, xd, yd, valid, in, G, G + (K + 1) * M, M, lane);
                }
                continue;
            }
            // the series ends in this slot: its points here join the sums (or, outside the interval, go one by one)
            bool added_old = false;
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                if (valid[e]) {
                    if (in[e]) { wa.add(mesh, xd[e], yd[e]); added_old = true; }
                    else scatter_point<K>(mesh, locate_interval(mesh, xd[e], LdgLoader()), xd[e], yd[e], G, G + (K + 1) * M, M);
                }
            }
            wa.dirty = wa.dirty || __any_sync(0xffffffffu, added_old);
            wa.flush(G, G + (K + 1) * M, M, lane);
            yy = warp_sum(yy);
            if (lane == 0) atomicAdd(G + (K + 2) * M, yy);
            yy = 0.0;
            // next series: that of the slot's last point (empty series are skipped by the search)
            const int64_t old_end = seg_end;
            seg = find_series(offsets, S, slot_last);
            const int64_t seg_begin = __ldg(offsets + seg);
            seg_end = __ldg(offsets + seg + 1);
            G = acc + seg * L;
            wa.cur = -1;
            wa.lo = INFINITY;
            wa.hi = -INFINITY;
            bool mine[VEC], none[VEC];
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                const int64_t q = p + e;
                mine[e] = q >= seg_begin && q < n;
                none[e] = false;
                if (mine[e]) yy = fma(yd[e], yd[e], yy);
                if (q >= old_end && q < seg_begin) {         // a series that lies wholly inside this slot
                    double* Gs = acc + find_series(offsets, S, q) * L;
                    scatter_point<K>(mesh, locate_interval(mesh, xd[e], LdgLoader()), xd[e], yd[e], Gs, Gs + (K + 1) * M, M);
                    atomicAdd(Gs + (K + 2) * M, yd[e] * yd[e]);
                }
            }
            // the lane holding the slot's last point has a point of the new series
            cross_interval<K, VEC>(wa, mesh, xd, yd, mine, none, G, G + (K + 1) * M, M, lane);
        }
    }
    wa.flush(G, G + (K + 1) * M, M, lane);
    if (seg >= 0) {
        yy = warp_sum(yy);
        if (lane == 0) atomicAdd(G + (K + 2) * M, yy);
    }
    for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < S; s += (int64_t)gridDim.x * blockDim.x)
        acc[s * L + L - 1] += (double)(__ldg(offsets + s + 1) - __ldg(offsets + s));
}

// ------------------------------------------------------------------------------------------------------------------
// accumulate for inputs in no particular order: bucket partition (partition.cuh), then per-unit shared-memory sort
// ------------------------------------------------------------------------------------------------------------------
constexpr int kUnitPoints1 = 4096;  // points per unit (2048-point units at three CTAs per SM spill and measured slower: 2.31 vs 2.13 ms)
constexpr int kUnitMargin = 2;      // intervals either side of a bucket the exact interval may fall into (a float32-built
                                    // mesh is not the uniform grid the bucket guess assumes); beyond: per-point REDs

template <class TX, class TY>
struct Points1D {
    const TX* x;
    const TY* y;
    const double* knots;
    int n_knots;
    int ipb;            // knot intervals per bucket
    Mesh mesh;
    __device__ __forceinline__ void init() { mesh = load_mesh(knots, n_knots); }
    __device__ __forceinline__ int guess(double xv) const {
        const double g = floor((xv - mesh.x0) * mesh.inv_delta);
        const int hi = n_knots - 2;
        return g < 0.0 ? 0 : (g > (double)hi ? hi : (int)g);
    }
    __device__ __forceinline__ int bucket(int64_t i) const { return guess((double)__ldg(x + i)) / ipb; }
    __device__ __forceinline__ void load(int64_t i, double (&v)[2]) const { v[0] = (double)__ldg(x + i); v[1] = (double)__ldg(y + i); }
    __device__ __forceinline__ int bucket_of(const double (&v)[2]) const { return guess(v[0]) / ipb; }
};

// One unit = up to kUnitPoints records of one bucket (= ipb consecutive knot intervals).  The CTA counting-sorts the unit
// by interval in shared memory (tau = t - 1/2 and y are what is staged), then groups of 8 lanes take whole intervals:
// the lanes of a group stride over the interval's run with the register moment sums of WarpAccum and the group flushes
// once per run (flush_groups).
template <int K, int THREADS>
__global__ void __launch_bounds__(THREADS, 2)
accum_1d_units_kernel(PartWork w, int64_t n, const double* __restrict__ knots, int n_knots, int ipb, int M,
                      double* __restrict__ G, double* __restrict__ b, double* __restrict__ scal) {
    constexpr int PER = kUnitPoints1 / THREADS;
    constexpr int kGroup = 8;
    constexpr int kWarps = THREADS / 32;
    extern __shared__ double s_dyn[];
    double* s_tau = s_dyn;                                            // [kUnitPoints1]
    double* s_y = s_tau + kUnitPoints1;                                // [kUnitPoints1]
    double* s_knots = s_y + kUnitPoints1;                              // [n_bins + 1]
    int* s_off = reinterpret_cast<int*>(s_knots + ipb + 2 * kUnitMargin + 1);   // [n_bins + 2]
    __shared__ UnitTable tab;
    __shared__ double s_yy[kWarps];
    __shared__ int s_wsum[kWarps];
    __shared__ int s_carry;
    const Mesh mesh = load_mesh(knots, n_knots);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_bins = ipb + 2 * kUnitMargin;
    const int last = n_knots - 2;                     // last interval
    const double* rx = w.rec;
    const double* ry = w.rec + n;
    tab.stage(w);
    __syncthreads();
    const int64_t n_slots = tab.n_slots();
    double yy = 0.0;
    WarpAccum<K> wa;
    wa.clear();
    for (int64_t u = blockIdx.x; u < n_slots; u += gridDim.x) {
        int bucket, count;
        int64_t first;
        if (!tab.find(u, kUnitPoints1, bucket, first, count)) continue;
        const int idx0 = bucket * ipb - kUnitMargin;          // interval of bin 0 (may be negative: those bins stay empty)
        const int jlo = idx0 < 0 ? -idx0 : 0;                 // bins [jlo, jhi] are real intervals
        const int jhi = (last - idx0 < n_bins - 1) ? last - idx0 : n_bins - 1;
        double xs[PER], ys[PER];
#pragma unroll
        for (int p = 0; p < PER; ++p) {
            const int q = p * THREADS + threadIdx.x;
            if (q < count) { xs[p] = __ldg(rx + first + q); ys[p] = __ldg(ry + first + q); }
        }
        for (int j = threadIdx.x; j <= n_bins; j += THREADS) {
            s_off[j] = 0;
            const int kn = idx0 + j;
            s_knots[j] = (kn >= 0 && kn < n_knots) ? __ldg(knots + kn) : 0.0;
        }
        __syncthreads();
        // exact interval (reference basis.py:58: largest idx with mesh[idx] < x) inside the staged window; count per bin
        // (bin j counts into s_off[j + 1])
        int bin[PER];
#pragma unroll
        for (int p = 0; p < PER; ++p) {
            const int q = p * THREADS + threadIdx.x;
            bin[p] = -1;
            if (q < count) {
                const double xv = xs[p];
                yy = fma(ys[p], ys[p], yy);
                const double g = floor((xv - mesh.x0) * mesh.inv_delta);
                int j = (g < (double)(idx0 + jlo)) ? jlo : (g > (double)(idx0 + jhi) ? jhi : (int)g - idx0);
                while (j > jlo && !(s_knots[j] < xv)) --j;
                while (j < jhi && s_knots[j + 1] < xv) ++j;
                const bool below = j == jlo && idx0 + jlo > 0 && !(s_knots[jlo] < xv);
                const bool above = j == jhi && idx0 + jhi < last && s_knots[jhi + 1] < xv;
                if (below || above) {       // outside the window (mesh far from uniform): per-point REDs
                    scatter_point<K>(mesh, locate_interval(mesh, xv, LdgLoader()), xv, ys[p], G, b, M);
                } else {
                    bin[p] = j;
                    atomicAdd(&s_off[j + 1], 1);
                }
            }
        }
        __syncthreads();
        // inclusive scan of s_off[1..n_bins] in place (s_off[j] becomes the first slot of bin j): chunks of THREADS + carry
        if (threadIdx.x == 0) s_carry = 0;
        __syncthreads();
        for (int base = 1; base <= n_bins; base += THREADS) {
            const int j = base + threadIdx.x;
            int v = j <= n_bins ? s_off[j] : 0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, v, o);
                if (lane >= o) v += t;
            }
            if (lane == 31) s_wsum[warp] = v;
            __syncthreads();
            int add = s_carry;
            for (int q = 0; q < warp; ++q) add += s_wsum[q];
            v += add;
            __syncthreads();
            if (j <= n_bins) s_off[j] = v;
            if (threadIdx.x == THREADS - 1) s_carry = v;
            __syncthreads();
        }
        // the placement advances s_off[j] from the start to the end of bin j, so afterwards bin j is
        // [j ? s_off[j - 1] : 0, s_off[j])
#pragma unroll
        for (int p = 0; p < PER; ++p) {
            if (bin[p] >= 0) {
                const int slot = atomicAdd(&s_off[bin[p]], 1);
                s_tau[slot] = fma(xs[p] - s_knots[bin[p]], mesh.inv_delta, -0.5);
                s_y[slot] = ys[p];
            }
        }
        __syncthreads();
        // kGroup lanes per interval, 32 / kGroup intervals per warp at a time
        for (int jb = warp * (32 / kGroup); jb < n_bins; jb += kWarps * (32 / kGroup)) {
            const int j = jb + lane / kGroup;
            int begin = 0, end = 0;
            if (j < n_bins) { begin = j ? s_off[j - 1] : 0; end = s_off[j]; }
            wa.cur = idx0 + j;
            for (int q = begin + (lane & (kGroup - 1)); q < end; q += kGroup) wa.add_tau(s_tau[q], s_y[q]);
            flush_groups<K, kGroup>(wa, end > begin, G, b, M, lane);
        }
        __syncthreads();
    }
    yy = warp_sum(yy);
    if (lane == 0) s_yy[warp] = yy;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
#pragma unroll
        for (int q = 0; q < kWarps; ++q) tot += s_yy[q];
        atomicAdd(scal, tot);
        if (blockIdx.x == 0) atomicAdd(scal + 1, (double)n);
    }
}

static size_t accum_1d_units_smem(int n_bins) { return (size_t)2 * kUnitPoints1 * 8 + (size_t)(n_bins + 1) * 8 + (size_t)(n_bins + 2) * 4; }

// Fraction of sampled neighbours (x[i], x[i+1]) that lie more than one knot interval apart: ~0 for time-series order,
// ~1 for shuffled input.  out[0] += jumps / samples.
template <class TX>
__global__ void __launch_bounds__(256) order_probe_1d_kernel(const TX* __restrict__ x, int64_t n, const double* __restrict__ knots,
                                                             int n_knots, int samples, double* __restrict__ out) {
    const Mesh mesh = load_mesh(knots, n_knots);
    int jumps = 0;
    for (int s = threadIdx.x; s < samples; s += blockDim.x) {
        const int64_t i = (int64_t)((double)s * (double)(n - 1) / (double)samples);
        const int a = locate_interval(mesh, (double)__ldg(x + i), LdgLoader()), c = locate_interval(mesh, (double)__ldg(x + i + 1), LdgLoader());
        jumps += (a - c > 1 || c - a > 1) ? 1 : 0;
    }
    jumps = __reduce_add_sync(0xffffffffu, jumps);
    if ((threadIdx.x & 31) == 0 && jumps) atomicAdd(out, (double)jumps / (double)samples);
}

// ------------------------------------------------------------------------------------------------------------------
// predictor
// ------------------------------------------------------------------------------------------------------------------
// Inside one knot interval the posterior mean is a polynomial of degree K and the variance one of degree 2K in
// tau = t - 1/2 (the same conversion tables as the accumulate, MomentCoef<K>): every lane caches the K+1 + 2K+1 coefficients
// of the interval it is in, so that a point of a time-ordered test set costs two Horner evaluations (3K+2 fp64
// instructions) and no gathers; lanes take consecutive pairs of points, loads and stores are fully coalesced 128-bit
// accesses.  A lane whose points jump between intervals (unordered test sets) evaluates pieces and window entries
// directly instead of refreshing its cache every time.  24 B of traffic per point.
// One lane's evaluator of the posterior (alpha, S, variance) with its interval cache; start() forgets the cache.
template <int K>
struct PredictPoint {
    const double* alpha;
    const double* S;
    double variance;
    int M;
    double cm[K + 1], cv[2 * K + 1];     // mean / variance polynomials (ascending powers of tau) of the cached interval
    int cur, since_refresh;
    double u, lo, hi;

    __device__ __forceinline__ void start(const double* alpha_, const double* S_, double variance_, int M_) {
        alpha = alpha_; S = S_; variance = variance_; M = M_;
        cur = -1; since_refresh = 1 << 20;
        u = 0.0; lo = INFINITY; hi = -INFINITY;
    }

    __device__ __forceinline__ void eval(const Mesh& mesh, double x, double& mu, double& vv) {
        const MomentCoef<K>& mc = g_moment_coef<K>;
        if (x > lo && x <= hi) {
            const double tau = fma(x - u, mesh.inv_delta, -0.5);
            double m = cm[K];
#pragma unroll
            for (int j = K - 1; j >= 0; --j) m = fma(m, tau, cm[j]);
            double v = cv[2 * K];
#pragma unroll
            for (int j = 2 * K - 1; j >= 0; --j) v = fma(v, tau, cv[j]);
            mu = m;
            vv = v;
            ++since_refresh;
            return;
        }
        const int idx = locate_interval(mesh, x, LdgLoader());
        const double ui = __ldg(mesh.knots + idx);
        if (since_refresh >= 8) {
            // the lane has been sitting in one interval: adopt the new one
            cur = idx;
            u = ui;
            lo = (idx == 0) ? -INFINITY : ui;
            hi = (idx == mesh.n_knots - 2) ? INFINITY : __ldg(mesh.knots + idx + 1);
#pragma unroll
            for (int j = 0; j <= K; ++j) cm[j] = 0.0;
#pragma unroll
            for (int j = 0; j <= 2 * K; ++j) cv[j] = 0.0;
#pragma unroll
            for (int r = 0; r <= K; ++r) {
                const double ar = __ldg(alpha + idx + r);
#pragma unroll
                for (int j = 0; j <= K; ++j) cm[j] = fma(mc.cb[r][j], ar, cm[j]);
#pragma unroll
                for (int q = 0; q <= r; ++q) {
                    const double sv = (q == r ? 1.0 : 2.0) * __ldg(S + (int64_t)(r - q) * M + idx + q);
#pragma unroll
                    for (int j = 0; j <= 2 * K; ++j) cv[j] = fma(mc.cg[tri_index(r, q)][j], sv, cv[j]);
                }
            }
            cv[0] += variance;
            since_refresh = 0;
            const double tau = fma(x - u, mesh.inv_delta, -0.5);
            double m = cm[K];
#pragma unroll
            for (int j = K - 1; j >= 0; --j) m = fma(m, tau, cm[j]);
            double v = cv[2 * K];
#pragma unroll
            for (int j = 2 * K - 1; j >= 0; --j) v = fma(v, tau, cv[j]);
            mu = m;
            vv = v;
            return;
        }
        // unordered points: direct evaluation from the pieces and the window entries
        since_refresh = 0;
        const double t = (x - ui) * mesh.inv_delta;
        double w[K + 1];
        bspline_pieces<K>(t, w);
        double m = 0.0, q = 0.0;
#pragma unroll
        for (int r = 0; r <= K; ++r) {
            m = fma(w[r], __ldg(alpha + idx + r), m);
            double row = 0.5 * w[r] * __ldg(S + idx + r);                       // diagonal counted once
#pragma unroll
            for (int sidx = 0; sidx < r; ++sidx) row = fma(w[sidx], __ldg(S + (int64_t)(r - sidx) * M + idx + sidx), row);
            q = fma(w[r], row, q);
        }
        mu = m;
        vv = variance + 2.0 * q;
    }
};

template <int K, int U, bool PREFETCH, int MINB>
__global__ void __launch_bounds__(256, MINB) predict_1d_kernel(const double* __restrict__ xs, int64_t n, const double* __restrict__ knots,
                                                         int n_knots, int M,
                                                         const double* __restrict__ alpha,
                                                         const double* __restrict__ S, double variance,
                                                         double* __restrict__ mean, double* __restrict__ var) {
    const Mesh mesh = load_mesh(knots, n_knots);
    const bool vec = ((reinterpret_cast<uintptr_t>(xs) | reinterpret_cast<uintptr_t>(mean) | reinterpret_cast<uintptr_t>(var)) & 15u) == 0;
    PredictPoint<K> pp;
    pp.start(alpha, S, variance, M);
    auto eval = [&](double x, double& mu, double& vv) { pp.eval(mesh, x, mu, vv); };

    if (vec) {
        // every CTA walks its own contiguous range of pairs in tiles of 256 * U, so that for an ordered test set a lane's
        // successive points are 2 * 256 * U apart and stay in one knot interval for many tiles
        const int64_t n_pairs = n >> 1;
        const int64_t per_cta = (n_pairs + gridDim.x - 1) / gridDim.x;
        const int64_t c_begin = blockIdx.x * per_cta, c_end = imin64(c_begin + per_cta, n_pairs);
        const double2* __restrict__ x2 = reinterpret_cast<const double2*>(xs);
        double2* __restrict__ m2 = reinterpret_cast<double2*>(mean);
        double2* __restrict__ v2 = reinterpret_cast<double2*>(var);
        // PREFETCH: the next tile's points are requested before the current tile is evaluated; the shipped instantiation
        // relies on four resident CTAs per SM instead (fewer registers; see the launch-shape note at asvgp_predict_1d)
        double2 xv[U];
        const uint64_t stream_policy = evict_first_policy();      // the test points are read once: keep alpha and the band in L2
        const int64_t step = (int64_t)blockDim.x * U;
        int64_t base = c_begin + threadIdx.x;
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int64_t i = base + j * (int64_t)blockDim.x;
            xv[j] = (i < c_end) ? ldg_stream2(xs + 2 * i, stream_policy) : make_double2(0.0, 0.0);
        }
        for (; base < c_end; base += step) {
            double2 xn[PREFETCH ? U : 1];
            if (PREFETCH) {
#pragma unroll
                for (int j = 0; j < U; ++j) {
                    const int64_t i = base + step + j * (int64_t)blockDim.x;
                    xn[j] = (i < c_end) ? ldg_stream2(xs + 2 * i, stream_policy) : make_double2(0.0, 0.0);
                }
            }
#pragma unroll
            for (int j = 0; j < U; ++j) {
                const int64_t i = base + j * (int64_t)blockDim.x;
                if (i >= c_end) break;
                double2 mo, vo;
                eval(xv[j].x, mo.x, vo.x);
                eval(xv[j].y, mo.y, vo.y);
                __stcs(m2 + i, mo);          // written once, never read back here
                __stcs(v2 + i, vo);
            }
            if (PREFETCH) {
#pragma unroll
                for (int j = 0; j < U; ++j) xv[j] = xn[j];
            } else {
#pragma unroll
                for (int j = 0; j < U; ++j) {
                    const int64_t i = base + step + j * (int64_t)blockDim.x;
                    xv[j] = (i < c_end) ? ldg_stream2(xs + 2 * i, stream_policy) : make_double2(0.0, 0.0);
                }
            }
        }
        if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) eval(__ldg(xs + n - 1), mean[n - 1], var[n - 1]);
    } else {
        const int64_t stride = (int64_t)gridDim.x * blockDim.x;
        for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) eval(__ldg(xs + i), mean[i], var[i]);
    }
}

// predict_1d_kernel's per-point evaluation for S posteriors at once: test points offsets[s] .. offsets[s+1] - 1 belong to series s
// (alpha + s M, S + s (K+1) M, variance[s]).  Every CTA walks a contiguous range with coalesced scalar accesses; a lane looks its
// series up again (and forgets its interval cache) whenever its point passes the current series' end.
template <int K>
__global__ void __launch_bounds__(256) predict_1d_segmented_kernel(const double* __restrict__ xs, int64_t n,
                                                                   const int64_t* __restrict__ offsets, int S,
                                                                   const double* __restrict__ knots, int n_knots, int M,
                                                                   const double* __restrict__ alpha, const double* __restrict__ Sb,
                                                                   const double* __restrict__ variance, double* __restrict__ mean,
                                                                   double* __restrict__ var) {
    const Mesh mesh = load_mesh(knots, n_knots);
    const int64_t per_cta = (n + gridDim.x - 1) / gridDim.x;
    const int64_t c_begin = blockIdx.x * per_cta, c_end = imin64(c_begin + per_cta, n);
    PredictPoint<K> pp;
    int64_t seg_end = -1;
    for (int64_t i = c_begin + threadIdx.x; i < c_end; i += blockDim.x) {
        if (i >= seg_end) {
            const int s = find_series(offsets, S, i);
            seg_end = __ldg(offsets + s + 1);
            pp.start(alpha + (int64_t)s * M, Sb + (int64_t)s * (K + 1) * M, __ldg(variance + s), M);
        }
        pp.eval(mesh, __ldg(xs + i), mean[i], var[i]);
    }
}

static int sm_count() {
    static int cached = 0;
    if (cached == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return 148;
        if (cudaDeviceGetAttribute(&cached, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) cached = 148;
    }
    return cached;
}

// CTA slots the streaming accumulate leaves free.  Its ranges are dealt statically (contiguous per CTA, so that ordered input
// meets few interval crossings), which makes it slow by a whole second wave as soon as ANY other kernel holds a few SMs; the
// bound's Kuu chain runs beside it on a cluster of 8 CTAs (banded_1d.cu, asvgp_kuu_chain_1d), each of which shares its SM with
// one CTA of this kernel: 4 SMs' worth of slots.  (What the chain really cost the accumulate was L2: see ldg_stream2.)
static int accum_sm_budget() {
    static int spare = -1;
    if (spare < 0) {
        const char* e = getenv("ASVGP_ACCUM_SPARE_SMS");
        spare = e ? atoi(e) : 4;
        if (spare < 0 || spare > sm_count() / 2) spare = 4;
    }
    return sm_count() - spare;
}

}  // namespace asvgp

using namespace asvgp;

#define ASVGP_DISPATCH_ORDER(order, CALL)          \
    switch (order) {                               \
        case 1: { constexpr int K = 1; CALL; } break; \
        case 2: { constexpr int K = 2; CALL; } break; \
        case 3: { constexpr int K = 3; CALL; } break; \
        case 4: { constexpr int K = 4; CALL; } break; \
        case 5: { constexpr int K = 5; CALL; } break; \
        case 6: { constexpr int K = 6; CALL; } break; \
        default:                                   \
            set_last_error("spline order %d not in 1..6", order); \
            return kBadArgument;                   \
    }

extern "C" int asvgp_basis_eval_1d(const double* x, int64_t n, const double* mesh, int n_knots, int order, int dx,
                                   const double* coef, int64_t* idx, double* vals, void* stream) {
    ASVGP_REQUIRE(n >= 0 && n_knots >= 2, "basis_eval_1d: n=%lld n_knots=%d", (long long)n, n_knots);
    ASVGP_REQUIRE(dx >= 0 && dx <= 3, "basis_eval_1d: dx=%d not in 0..3 (reference basis.py:61-70)", dx);
    ASVGP_REQUIRE(dx == 0 || coef != nullptr, "basis_eval_1d: dx>0 needs the piece coefficient table");
    if (n == 0) return kOk;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int blocks = (int)std::min<int64_t>((n + 255) / 256, (int64_t)sm_count() * 8);
    ASVGP_DISPATCH_ORDER(order, (basis_eval_1d_kernel<K><<<blocks, 256, 0, st>>>(x, n, mesh, n_knots, dx, coef, idx, vals))); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

template <class TX, class TY>
static int launch_accum_1d(const TX* x, const TY* y, int64_t n, const double* mesh, int n_knots, int order, double* acc,
                           cudaStream_t st) {
    const int M = n_knots + order - 1;
    double* G = acc;
    double* b = acc + (int64_t)(order + 1) * M;
    double* scal = b + M;
    const bool vec = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15u) == 0;
    constexpr int VV = (sizeof(TX) == 8 && sizeof(TY) == 8) ? 2 : 4;      // points per slot of the vector path
    const int64_t per_tile = 32 * (vec ? (int64_t)accum_unroll<VV, TX, TY>() * VV : (int64_t)accum_unroll<1, TX, TY>());
    const int64_t n_tiles = (n + per_tile - 1) / per_tile;
    // (tools/accum_sweep.py: 2 and 4 CTAs' worth of ranges per SM both give 0.258 ms at N = 1e8; 3, 8, 16 are slower)
    const int blocks = (int)std::min<int64_t>((n_tiles + 7) / 8, (int64_t)accum_sm_budget() * 2);
    if (vec) {
        ASVGP_DISPATCH_ORDER(order, (accum_1d_kernel<K, VV, TX, TY><<<blocks, kAccumThreads, 0, st>>>(x, y, n, mesh, n_knots, M, G, b, scal))); ASVGP_LAUNCHED();
    } else {
        ASVGP_DISPATCH_ORDER(order, (accum_1d_kernel<K, 1, TX, TY><<<blocks, kAccumThreads, 0, st>>>(x, y, n, mesh, n_knots, M, G, b, scal))); ASVGP_LAUNCHED();
    }
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

extern "C" int asvgp_accum_1d_typed(const void* x, int x_type, const void* y, int y_type, int64_t n, const double* mesh,
                                    int n_knots, int order, double* acc, void* stream) {
    ASVGP_REQUIRE_TYPES("accum_1d", x_type, y_type);
    ASVGP_REQUIRE(n >= 0 && n_knots >= 2, "accum_1d: n=%lld n_knots=%d", (long long)n, n_knots);
    ASVGP_REQUIRE(order >= 1 && order <= kMaxOrder, "accum_1d: spline order %d not in 1..6", order);
    if (n == 0) return kOk;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    return with_elem_types(x_type, y_type, [&](auto tx, auto ty) -> int {
        using TX = typename decltype(tx)::type;
        using TY = typename decltype(ty)::type;
        return launch_accum_1d(static_cast<const TX*>(x), static_cast<const TY*>(y), n, mesh, n_knots, order, acc, st);
    });
}

extern "C" int asvgp_accum_1d(const double* x, const double* y, int64_t n, const double* mesh, int n_knots, int order,
                              double* acc, void* stream) {
    return asvgp_accum_1d_typed(x, ASVGP_F64, y, ASVGP_F64, n, mesh, n_knots, order, acc, stream);
}

template <class TX, class TY>
static int launch_accum_1d_segmented(const TX* x, const TY* y, int64_t n, const int64_t* offsets, int S, const double* mesh,
                                     int n_knots, int order, double* acc, cudaStream_t st) {
    const int M = n_knots + order - 1;
    const bool vec = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15u) == 0;
    constexpr int VV = (sizeof(TX) == 8 && sizeof(TY) == 8) ? 2 : 4;
    const int64_t per_tile = 32 * (vec ? (int64_t)accum_unroll<VV, TX, TY>() * VV : (int64_t)accum_unroll<1, TX, TY>());
    const int64_t n_tiles = (n + per_tile - 1) / per_tile;
    // the grid of launch_accum_1d; at least one CTA, whose grid-stride loop writes the counts
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((n_tiles + 7) / 8, (int64_t)accum_sm_budget() * 2));
    if (vec) {
        ASVGP_DISPATCH_ORDER(order, (accum_1d_segmented_kernel<K, VV, TX, TY><<<blocks, kAccumThreads, 0, st>>>(x, y, n, offsets, S, mesh, n_knots, M, acc))); ASVGP_LAUNCHED();
    } else {
        ASVGP_DISPATCH_ORDER(order, (accum_1d_segmented_kernel<K, 1, TX, TY><<<blocks, kAccumThreads, 0, st>>>(x, y, n, offsets, S, mesh, n_knots, M, acc))); ASVGP_LAUNCHED();
    }
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

extern "C" int asvgp_accum_1d_segmented_typed(const void* x, int x_type, const void* y, int y_type, int64_t n, const int64_t* offsets,
                                              int S, const double* mesh, int n_knots, int order, double* acc, void* stream) {
    ASVGP_REQUIRE_TYPES("accum_1d_segmented", x_type, y_type);
    ASVGP_REQUIRE(S >= 1, "accum_1d_segmented: S=%d must be at least 1", S);
    ASVGP_REQUIRE(n >= 0 && n_knots >= 2, "accum_1d_segmented: n=%lld n_knots=%d", (long long)n, n_knots);
    ASVGP_REQUIRE(order >= 1 && order <= kMaxOrder, "accum_1d_segmented: spline order %d not in 1..6", order);
    ASVGP_REQUIRE(offsets != nullptr, "accum_1d_segmented: offsets is NULL");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    return with_elem_types(x_type, y_type, [&](auto tx, auto ty) -> int {
        using TX = typename decltype(tx)::type;
        using TY = typename decltype(ty)::type;
        return launch_accum_1d_segmented(static_cast<const TX*>(x), static_cast<const TY*>(y), n, offsets, S, mesh, n_knots, order, acc, st);
    });
}

extern "C" int64_t asvgp_accum_1d_binned_work_bytes(int64_t n) { return PartWork::bytes(n < 0 ? 0 : n, 2); }

extern "C" int asvgp_order_probe_1d_typed(const void* x, int x_type, int64_t n, const double* mesh, int n_knots, double* out,
                                          void* stream) {
    ASVGP_REQUIRE(valid_elem_type(x_type), "order_probe_1d: element type %d (0 = float64, 1 = float32)", x_type);
    ASVGP_REQUIRE(n >= 0 && n_knots >= 2 && out != nullptr, "order_probe_1d: n=%lld n_knots=%d", (long long)n, n_knots);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ASVGP_CUDA_OK(cudaMemsetAsync(out, 0, sizeof(double), st));
    if (n < 2) return kOk;
    const int samples = (int)std::min<int64_t>(n - 1, 4096);
    if (x_type == ASVGP_F32) order_probe_1d_kernel<<<1, 256, 0, st>>>(static_cast<const float*>(x), n, mesh, n_knots, samples, out);
    else order_probe_1d_kernel<<<1, 256, 0, st>>>(static_cast<const double*>(x), n, mesh, n_knots, samples, out);
    ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

extern "C" int asvgp_order_probe_1d(const double* x, int64_t n, const double* mesh, int n_knots, double* out, void* stream) {
    return asvgp_order_probe_1d_typed(x, ASVGP_F64, n, mesh, n_knots, out, stream);
}

template <int K>
static int launch_accum_1d_units(const PartWork& w, int64_t n, const double* mesh, int n_knots, int ipb, int M, double* G,
                                 double* b, double* scal, cudaStream_t st) {
    constexpr int THREADS = 256;         // (512 threads at 64 registers spill the moment sums and measured no faster)
    const size_t smem = accum_1d_units_smem(ipb + 2 * kUnitMargin);
    ASVGP_CUDA_OK(cudaFuncSetAttribute(accum_1d_units_kernel<K, THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    ASVGP_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, accum_1d_units_kernel<K, THREADS>, THREADS, smem));
    const int64_t max_units = n / kUnitPoints1 + kPartBuckets;
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(max_units, (int64_t)sm_count() * std::max(per_sm, 1)));
    accum_1d_units_kernel<K, THREADS><<<blocks, THREADS, smem, st>>>(w, n, mesh, n_knots, ipb, M, G, b, scal); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

extern "C" int asvgp_accum_1d_binned_typed(const void* x, int x_type, const void* y, int y_type, int64_t n, const double* mesh,
                                           int n_knots, int order, double* acc, void* work, int64_t work_bytes, void* stream) {
    ASVGP_REQUIRE_TYPES("accum_1d_binned", x_type, y_type);
    ASVGP_REQUIRE(n >= 0 && n_knots >= 2, "accum_1d_binned: n=%lld n_knots=%d", (long long)n, n_knots);
    ASVGP_REQUIRE(order >= 1 && order <= kMaxOrder, "accum_1d_binned: spline order %d not in 1..6", order);
    const int n_int = n_knots - 1;
    const int ipb = (n_int + kPartBuckets - 1) / kPartBuckets;
    if (ipb + 2 * kUnitMargin > kUnitMaxBins)  // more than ~2^20 knot intervals: the general kernel handles any order
        return asvgp_accum_1d_typed(x, x_type, y, y_type, n, mesh, n_knots, order, acc, stream);
    ASVGP_REQUIRE(work != nullptr && work_bytes >= PartWork::bytes(n, 2), "accum_1d_binned: work_bytes=%lld < %lld",
                  (long long)work_bytes, (long long)PartWork::bytes(n, 2));
    if (n == 0) return kOk;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int M = n_knots + order - 1;
    double* G = acc;
    double* b = acc + (int64_t)(order + 1) * M;
    double* scal = b + M;
    const PartWork w = PartWork::carve(work);
    ASVGP_CUDA_OK(cudaMemsetAsync(w.count, 0, kPartBuckets * sizeof(u64), st));
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((n + kPartTile - 1) / kPartTile, (int64_t)sm_count() * 2));
    // the partition reads the points in their own types and writes float64 records: the units kernel is type-free
    const int prc = with_elem_types(x_type, y_type, [&](auto tx, auto ty) -> int {
        using TX = typename decltype(tx)::type;
        using TY = typename decltype(ty)::type;
        Points1D<TX, TY> src;
        src.x = static_cast<const TX*>(x); src.y = static_cast<const TY*>(y); src.knots = mesh; src.n_knots = n_knots; src.ipb = ipb;
        ASVGP_CUDA_OK((launch_partition<Points1D<TX, TY>, 2>(src, n, w, kUnitPoints1, blocks, st)));
        return kOk;
    });
    if (prc != kOk) return prc;
    int rc = kOk;
    ASVGP_DISPATCH_ORDER(order, (rc = launch_accum_1d_units<K>(w, n, mesh, n_knots, ipb, M, G, b, scal, st)));
    return rc;
}

extern "C" int asvgp_accum_1d_binned(const double* x, const double* y, int64_t n, const double* mesh, int n_knots, int order,
                                     double* acc, void* work, int64_t work_bytes, void* stream) {
    return asvgp_accum_1d_binned_typed(x, ASVGP_F64, y, ASVGP_F64, n, mesh, n_knots, order, acc, work, work_bytes, stream);
}

extern "C" int asvgp_predict_1d(const double* xnew, int64_t n, const double* mesh, int n_knots, int order,
                                const double* alpha, const double* S_band, double variance, double* mean, double* var,
                                void* stream) {
    ASVGP_REQUIRE(n >= 0 && n_knots >= 2, "predict_1d: n=%lld n_knots=%d", (long long)n, n_knots);
    if (n == 0) return kOk;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int M = n_knots + order - 1;
    // Launch shape (tools/predict_1d_sweep.py, 1e8 sorted points): 64 registers / 4 CTAs per SM with two pairs in flight per
    // thread and MANY short CTA ranges — 0.47 ms = 5.1 TB/s, the ceiling of a 1 : 2 read : write stream on this part
    // (tools/microbench/rw12_bench.cu: 5.4 TB/s) — against 0.69 ms for 4 prefetched pairs at 80+ registers on 4 CTAs per SM.
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((n + 4095) / 4096, (int64_t)sm_count() * 128));
    ASVGP_DISPATCH_ORDER(order, (predict_1d_kernel<K, 2, false, 4><<<blocks, 256, 0, st>>>(xnew, n, mesh, n_knots, M, alpha, S_band, variance, mean, var)));
    ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

extern "C" int asvgp_predict_1d_segmented(const double* xnew, int64_t n, const int64_t* offsets_new, int S, const double* mesh,
                                          int n_knots, int order, const double* alpha, const double* S_band, const double* variance,
                                          double* mean, double* var, void* stream) {
    ASVGP_REQUIRE(S >= 1, "predict_1d_segmented: S=%d must be at least 1", S);
    ASVGP_REQUIRE(n >= 0 && n_knots >= 2, "predict_1d_segmented: n=%lld n_knots=%d", (long long)n, n_knots);
    ASVGP_REQUIRE(order >= 1 && order <= kMaxOrder, "predict_1d_segmented: spline order %d not in 1..6", order);
    ASVGP_REQUIRE(offsets_new != nullptr, "predict_1d_segmented: offsets_new is NULL");
    if (n == 0) return kOk;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int M = n_knots + order - 1;
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((n + 4095) / 4096, (int64_t)sm_count() * 128));
    ASVGP_DISPATCH_ORDER(order, (predict_1d_segmented_kernel<K><<<blocks, 256, 0, st>>>(xnew, n, offsets_new, S, mesh, n_knots, M, alpha,
                                                                                     S_band, variance, mean, var)));
    ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}
