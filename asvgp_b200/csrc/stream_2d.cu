// Streaming 2-D (Kronecker) kernels: fused Gram/projection accumulation and posterior predictor.
//
//   asvgp_accum_2d   <- GPR_kron.__init__ precompute: per-dimension make_Kuf, kron.make_kvs_sparse (row-wise
//                       Khatri-Rao), Kuf @ y, Kuf @ Kuf.T           (reference asvgp/gpr.py:268-274, kronecker.py:7-33)
//   asvgp_predict_2d <- GPR_kron.predict_f / predict_f_sparse       (reference asvgp/gpr.py:310-359)
//
// accum_2d design (DESIGN.md §4.3).  A point in cell (c1, c2) adds w w^T with w = a (x) b, a = pieces(t1),
// b = pieces(t2): (k+1)^2 ((k+1)^2 + 1)/2 = 136 products for k = 3 — too many accumulators for one thread, and the
// kernel would sit far above the fp64 ridge.  But every product a_r a_s b_u b_v is a polynomial of degree 2k in t1 and
// in t2, so all of them live in the (2k+1)^2-dimensional span of
//        beta_p(t1) beta_q(t2),   beta_p(t) = t^p (1-t)^(2k-p),
// and expand in it with NON-NEGATIVE coefficients (B-spline pieces have non-negative Bezier coefficients), i.e. without
// cancellation.  So each thread keeps (2k+1)^2 + (k+1)^2 = 65 moment sums (k = 3) in registers for the cell it is in,
// one FMA per moment per point, and flushes them to a per-cell moment table (fp64 RED, L2 resident) when its points
// move to another cell.  A second, tiny kernel expands the moment table into the Gram stencil and the projection.
// Every thread walks its own contiguous slice of the points, so raster-ordered data (x1 slow) gives runs of
// ~n2/(m2-k) points per flush; any order gives the right answer.
// X and y may each be float32 or float64 (asvgp_accum_2d_typed): every kernel that reads points is templated on the two
// element types and converts each loaded value to double in registers (12 B per point for float32 data instead of 24).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>

#include "async_copy.cuh"
#include "common.cuh"
#include "partition.cuh"
#include "../../include/asvgp_b200.h"

namespace asvgp {

struct LdgLoader2 {
    __device__ __forceinline__ double operator()(const double* p) const { return __ldg(p); }
};
struct PlainLoader2 {         // generic load: the knots may sit in shared memory
    __device__ __forceinline__ double operator()(const double* p) const { return *p; }
};

__device__ __forceinline__ Mesh load_mesh2(const double* knots, int n_knots) {
    Mesh m;
    m.knots = knots;
    m.n_knots = n_knots;
    m.x0 = __ldg(knots);
    m.inv_delta = 1.0 / (__ldg(knots + 1) - m.x0);
    return m;
}

// Loads of the training points, which are float64 or float32 (X and y independently): every value is converted to double
// in registers (exact), so everything after the load is the float64 code.
__device__ __forceinline__ double ldg_d(const double* p) { return __ldg(p); }
__device__ __forceinline__ double ldg_d(const float* p) { return (double)__ldg(p); }
// point i (x1, x2) of a row-major [n, 2] array
__device__ __forceinline__ double2 ldg_point(const double* X, int64_t i) { return __ldg(reinterpret_cast<const double2*>(X) + i); }
__device__ __forceinline__ double2 ldg_point(const float* X, int64_t i) {
    const float2 p = __ldg(reinterpret_cast<const float2*>(X) + i);
    return make_double2(p.x, p.y);
}
// targets i and i + 1, i even (one 16-byte / 8-byte load)
__device__ __forceinline__ double2 ldg_pair(const double* y, int64_t i) { return __ldg(reinterpret_cast<const double2*>(y + i)); }
__device__ __forceinline__ double2 ldg_pair(const float* y, int64_t i) {
    const float2 p = __ldg(reinterpret_cast<const float2*>(y + i));
    return make_double2(p.x, p.y);
}

struct Interval {            // cached knot interval of one dimension
    int idx;
    double u, lo, hi;
    __device__ __forceinline__ void reset() { idx = -1; u = 0.0; lo = INFINITY; hi = -INFINITY; }
    __device__ __forceinline__ bool inside(double x) const { return x > lo && x <= hi; }
    __device__ __forceinline__ void set(const Mesh& mesh, int i) { set(mesh, i, LdgLoader2()); }
    template <class LoadFn>
    __device__ __forceinline__ void set(const Mesh& mesh, int i, LoadFn load) {
        idx = i;
        u = load(mesh.knots + i);
        lo = (i == 0) ? -INFINITY : u;
        hi = (i == mesh.n_knots - 2) ? INFINITY : load(mesh.knots + i + 1);
    }
};

template <int K> struct Moments {
    static constexpr int NB = 2 * K + 1;            // Bernstein-type functions per dimension for the Gram part
    static constexpr int NY = K + 1;                // ... for the projection part
    static constexpr int kGram = NB * NB;
    static constexpr int kProj = NY * NY;
    static constexpr int kAll = kGram + kProj;      // doubles per cell in the moment table
};

// powers t^0..t^N and (1-t)^0..(1-t)^N
template <int N>
__device__ __forceinline__ void powers(double t, double (&tp)[N + 1], double (&up)[N + 1]) {
    const double u = 1.0 - t;
    tp[0] = 1.0; up[0] = 1.0;
#pragma unroll
    for (int i = 1; i <= N; ++i) { tp[i] = tp[i - 1] * t; up[i] = up[i - 1] * u; }
}

// Thread-private accumulation over a contiguous slice of points.  [P0, P1) is the range of the dim-1 moment index
// this launch handles (register budget: one launch for k <= 3, split launches for k >= 4); WITH_Y: also the
// projection moments, sum y^2 and the count.
template <int K, int P0, int P1, bool WITH_Y, class TX, class TY>
__global__ void __launch_bounds__(256, 1)
accum_2d_kernel(const TX* __restrict__ X, const TY* __restrict__ y, int64_t n,
                const double* __restrict__ knots1, int nk1, const double* __restrict__ knots2, int nk2,
                double* __restrict__ cellmom, double* __restrict__ scal, const int* __restrict__ select, int want) {
    if (select != nullptr && *select != want) return;
    using Mo = Moments<K>;
    constexpr int NB = Mo::NB, NY = Mo::NY;
    constexpr int NP = P1 - P0;
    const Mesh mesh1 = load_mesh2(knots1, nk1), mesh2 = load_mesh2(knots2, nk2);
    const int nc2 = nk2 - 1;

    const int64_t n_threads = (int64_t)gridDim.x * blockDim.x;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t per = (n + n_threads - 1) / n_threads;
    per = (per + 1) & ~(int64_t)1;                                  // even: y is read two points at a time
    const int64_t begin = tid * per < n ? tid * per : n;
    const int64_t end = begin + per < n ? begin + per : n;

    double acc[NP * NB];
    double accy[WITH_Y ? NY * NY : 1];
#pragma unroll
    for (int i = 0; i < NP * NB; ++i) acc[i] = 0.0;
#pragma unroll
    for (int i = 0; i < (WITH_Y ? NY * NY : 1); ++i) accy[i] = 0.0;
    double yy = 0.0;
    Interval i1, i2;
    i1.reset(); i2.reset();
    bool dirty = false;

    auto flush = [&]() {
        if (dirty) {
            double* dst = cellmom + ((int64_t)i1.idx * nc2 + i2.idx) * Mo::kAll;
#pragma unroll
            for (int p = 0; p < NP; ++p)
#pragma unroll
                for (int q = 0; q < NB; ++q) {
                    atomicAdd(dst + (P0 + p) * NB + q, acc[p * NB + q]);
                    acc[p * NB + q] = 0.0;
                }
            if (WITH_Y) {
#pragma unroll
                for (int i = 0; i < NY * NY; ++i) { atomicAdd(dst + Mo::kGram + i, accy[i]); accy[i] = 0.0; }
            }
            dirty = false;
        }
    };
    auto add = [&](double x1, double x2, double yv) {
        if (!(i1.inside(x1) && i2.inside(x2))) {
            flush();
            if (!i1.inside(x1)) i1.set(mesh1, locate_interval(mesh1, x1, LdgLoader2()));
            if (!i2.inside(x2)) i2.set(mesh2, locate_interval(mesh2, x2, LdgLoader2()));
        }
        const double t1 = (x1 - i1.u) * mesh1.inv_delta, t2 = (x2 - i2.u) * mesh2.inv_delta;
        double tp1[2 * K + 1], up1[2 * K + 1], tp2[2 * K + 1], up2[2 * K + 1];
        powers<2 * K>(t1, tp1, up1);
        powers<2 * K>(t2, tp2, up2);
        double b2[NB];
#pragma unroll
        for (int q = 0; q < NB; ++q) b2[q] = tp2[q] * up2[2 * K - q];
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            const double b1 = tp1[P0 + p] * up1[2 * K - (P0 + p)];
#pragma unroll
            for (int q = 0; q < NB; ++q) acc[p * NB + q] = fma(b1, b2[q], acc[p * NB + q]);
        }
        if (WITH_Y) {
            double g2[NY];
#pragma unroll
            for (int q = 0; q < NY; ++q) g2[q] = tp2[q] * up2[K - q];
#pragma unroll
            for (int p = 0; p < NY; ++p) {
                const double g1 = yv * (tp1[p] * up1[K - p]);
#pragma unroll
                for (int q = 0; q < NY; ++q) accy[p * NY + q] = fma(g1, g2[q], accy[p * NY + q]);
            }
            yy = fma(yv, yv, yy);
        }
        dirty = true;
    };

    // X is row-major [n, 2]: one 16-byte (float32: 8-byte) load per point; begin is even so y pairs are aligned too
    int64_t i = begin;
    for (; i + 4 <= end; i += 4) {
        const double2 pa = ldg_point(X, i), pb = ldg_point(X, i + 1), pc = ldg_point(X, i + 2), pd = ldg_point(X, i + 3);
        double2 ya = make_double2(0.0, 0.0), yb = ya;
        if (WITH_Y) {
            ya = ldg_pair(y, i);
            yb = ldg_pair(y, i + 2);
        }
        add(pa.x, pa.y, ya.x);
        add(pb.x, pb.y, ya.y);
        add(pc.x, pc.y, yb.x);
        add(pd.x, pd.y, yb.y);
    }
    for (; i < end; ++i) {
        const double2 pa = ldg_point(X, i);
        add(pa.x, pa.y, WITH_Y ? ldg_d(y + i) : 0.0);
    }
    flush();

    if (WITH_Y) {
        __shared__ double s_yy[8];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) yy += __shfl_xor_sync(0xffffffffu, yy, o);
        if ((threadIdx.x & 31) == 0) s_yy[threadIdx.x >> 5] = yy;
        __syncthreads();
        if (threadIdx.x == 0) {
            double tot = 0.0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += s_yy[w];
            atomicAdd(scal, tot);
            if (blockIdx.x == 0) atomicAdd(scal + 1, (double)n);
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// "run" path for gridded input (raster order: consecutive points share x1 bit-for-bit, as a flattened lon/lat mesh
// does).  For a run of points with the same x1 inside one cell the dim-1 factors are constant, so
//     mom[p][q] += beta_p(t1) * sum_n beta_q(t2_n),      ymom[p][q] += gamma_p(t1) * sum_n y_n gamma_q(t2_n):
// per point only the (2k+1) + (k+1) dim-2 sums are updated (~35 fp64 instructions for k = 3 instead of ~120), and
// the outer product with the dim-1 factors happens once per run, straight into the L2-resident moment table.
// A thread keeps ~4k+4 sums instead of (2k+1)^2 + (k+1)^2, which triples the occupancy.  Any input is still
// handled correctly (a run may have length 1); asvgp_accum_2d picks this kernel when a probe finds the input
// gridded.
// ------------------------------------------------------------------------------------------------------------------
template <int K, class TX, class TY>
__global__ void __launch_bounds__(256, 2)
accum_2d_run_kernel(const TX* __restrict__ X, const TY* __restrict__ y, int64_t n,
                    const double* __restrict__ knots1, int nk1, const double* __restrict__ knots2, int nk2,
                    double* __restrict__ cellmom, double* __restrict__ scal, const int* __restrict__ select,
                    int want) {
    if (select != nullptr && *select != want) return;
    using Mo = Moments<K>;
    constexpr int NB = Mo::NB, NY = Mo::NY;
    const Mesh mesh1 = load_mesh2(knots1, nk1), mesh2 = load_mesh2(knots2, nk2);
    const int nc2 = nk2 - 1;

    const int64_t n_threads = (int64_t)gridDim.x * blockDim.x;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t per = (n + n_threads - 1) / n_threads;
    per = (per + 3) & ~(int64_t)3;                                  // groups of four points, y read as two double2
    const int64_t begin = tid * per < n ? tid * per : n;
    const int64_t end = begin + per < n ? begin + per : n;

    double s[NB], sy[NY], b1[NB], g1[NY];
#pragma unroll
    for (int i = 0; i < NB; ++i) { s[i] = 0.0; b1[i] = 0.0; }
#pragma unroll
    for (int i = 0; i < NY; ++i) { sy[i] = 0.0; g1[i] = 0.0; }
    double yy = 0.0;
    long long cur_x1 = 0;              // bit pattern of the run's x1
    bool have_x1 = false, dirty = false;
    Interval i1, i2;
    i1.reset(); i2.reset();

    auto flush = [&]() {
        if (dirty) {
            double* dst = cellmom + ((int64_t)i1.idx * nc2 + i2.idx) * Mo::kAll;
#pragma unroll
            for (int p = 0; p < NB; ++p)
#pragma unroll
                for (int q = 0; q < NB; ++q) atomicAdd(dst + p * NB + q, b1[p] * s[q]);
#pragma unroll
            for (int p = 0; p < NY; ++p)
#pragma unroll
                for (int q = 0; q < NY; ++q) atomicAdd(dst + Mo::kGram + p * NY + q, g1[p] * sy[q]);
#pragma unroll
            for (int q = 0; q < NB; ++q) s[q] = 0.0;
#pragma unroll
            for (int q = 0; q < NY; ++q) sy[q] = 0.0;
            dirty = false;
        }
    };
    auto add = [&](double x1, double x2, double yv) {
        const long long bits = __double_as_longlong(x1);
        const bool same_x1 = have_x1 && bits == cur_x1;
        if (!(same_x1 && i2.inside(x2))) {
            flush();
            if (!same_x1) {
                if (!i1.inside(x1)) i1.set(mesh1, locate_interval(mesh1, x1, LdgLoader2()));
                const double t1 = (x1 - i1.u) * mesh1.inv_delta;
                double tp[2 * K + 1], up[2 * K + 1];
                powers<2 * K>(t1, tp, up);
#pragma unroll
                for (int p = 0; p < NB; ++p) b1[p] = tp[p] * up[2 * K - p];
#pragma unroll
                for (int p = 0; p < NY; ++p) g1[p] = tp[p] * up[K - p];
                cur_x1 = bits;
                have_x1 = true;
            }
            if (!i2.inside(x2)) i2.set(mesh2, locate_interval(mesh2, x2, LdgLoader2()));
        }
        const double t2 = (x2 - i2.u) * mesh2.inv_delta;
        double tp[2 * K + 1], up[2 * K + 1];
        powers<2 * K>(t2, tp, up);
#pragma unroll
        for (int q = 0; q < NB; ++q) s[q] += tp[q] * up[2 * K - q];
#pragma unroll
        for (int q = 0; q < NY; ++q) sy[q] = fma(yv, tp[q] * up[K - q], sy[q]);
        yy = fma(yv, yv, yy);
        dirty = true;
    };

    // X is row-major [n, 2]: one 16-byte (float32: 8-byte) load per point; begin is a multiple of 4 so y pairs are aligned.
    // The next group's loads are issued before the current group is processed.
    const int64_t n_full = begin + ((end - begin) & ~(int64_t)3);
    double2 pa, pb, pc, pd, ya, yb;
    int64_t i = begin;
    if (i < n_full) {
        pa = ldg_point(X, i); pb = ldg_point(X, i + 1); pc = ldg_point(X, i + 2); pd = ldg_point(X, i + 3);
        ya = ldg_pair(y, i); yb = ldg_pair(y, i + 2);
    }
    for (; i < n_full; i += 4) {
        const double2 ca = pa, cb = pb, cc = pc, cd = pd, cya = ya, cyb = yb;
        if (i + 4 < n_full) {
            pa = ldg_point(X, i + 4); pb = ldg_point(X, i + 5); pc = ldg_point(X, i + 6); pd = ldg_point(X, i + 7);
            ya = ldg_pair(y, i + 4); yb = ldg_pair(y, i + 6);
        }
        add(ca.x, ca.y, cya.x);
        add(cb.x, cb.y, cya.y);
        add(cc.x, cc.y, cyb.x);
        add(cd.x, cd.y, cyb.y);
    }
    for (; i < end; ++i) {
        const double2 p = ldg_point(X, i);
        add(p.x, p.y, ldg_d(y + i));
    }
    flush();

    __shared__ double s_yy[8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) yy += __shfl_xor_sync(0xffffffffu, yy, o);
    if ((threadIdx.x & 31) == 0) s_yy[threadIdx.x >> 5] = yy;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += s_yy[w];
        atomicAdd(scal, tot);
        if (blockIdx.x == 0) atomicAdd(scal + 1, (double)n);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// "raster" path: the input is a flattened n1 x n2 mesh (x1 slow; every n2 consecutive points share x1 bit for bit).
// The index space is tiled as (32 rows) x (column segment); the lanes of a warp walk 32 different rows in lock-step,
// so on a separable mesh all lanes cross a knot of dimension 2 at the same step and the flush is convergent and
// cooperative: the 32 per-lane dim-2 sums go through shared memory, are contracted with the per-lane dim-1 factors and
// leave as THREE fp64 REDs per lane per (cell, 32 rows) — 32x fewer atomics than one flush per lane.  Each lane streams
// its own row with 256-bit loads (LDG.E.256), the next group of four points in flight while the current one is
// processed.  Correctness never depends on the mesh being regular: every lane handles exactly the index range of its
// row tile, flushing whenever ITS x1 or ITS cell changes (a warp vote makes the others flush early with it).
// ------------------------------------------------------------------------------------------------------------------
struct ProbeResult {      // lives in the trailing slot of the moment table (two ints)
    int select;           // 0 general, 1 x1-run, 2 raster (per-point loads), 3 raster (256-bit loads), 4 separable raster
    int n2;               // row length of the raster
};

// Bulk L2 prefetch (UBLKPF.L2): pulls `bytes` (multiple of 16, 16-byte aligned start) from DRAM into L2 without occupying
// registers or shared memory.  The streaming kernels run at (bytes in flight) / (loaded DRAM latency ~2 us); prefetching a
// block ahead turns their register-staged loads into L2 hits.
__device__ __forceinline__ void prefetch_l2_bulk(const void* p, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
__device__ __forceinline__ void prefetch_l2_span(const double* first, int64_t n_doubles) {
    // widen [first, first + n) to 16-byte boundaries
    const uintptr_t a = reinterpret_cast<uintptr_t>(first) & ~(uintptr_t)15;
    const uintptr_t e = (reinterpret_cast<uintptr_t>(first + n_doubles) + 15) & ~(uintptr_t)15;
    prefetch_l2_bulk(reinterpret_cast<const void*>(a), (uint32_t)(e - a));
}

__device__ __forceinline__ void ldg256(const double* p, double (&v)[4]) {
    asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(v[0]), "=d"(v[1]), "=d"(v[2]), "=d"(v[3]) : "l"(p));
}
// four consecutive values as double: one 256-bit load of float64, one 128-bit load of float32
__device__ __forceinline__ void ldg4(const double* p, double (&v)[4]) { ldg256(p, v); }
__device__ __forceinline__ void ldg4(const float* p, double (&v)[4]) {
    const float4 f = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
}

constexpr int kRasterWarps = 8;          // 256 threads, two CTAs per SM (<= 128 registers per thread): occupancy beats
                                         // a deeper register-staged prefetch here (measured: 6 warps x 8-point groups was slower)

template <int K, bool VEC256, class TX, class TY>
__global__ void __launch_bounds__(kRasterWarps * 32, 2)
accum_2d_raster_kernel(const TX* __restrict__ X, const TY* __restrict__ y, int64_t n,
                       const double* __restrict__ knots1, int nk1, const double* __restrict__ knots2, int nk2,
                       double* __restrict__ cellmom, double* __restrict__ scal, const ProbeResult* __restrict__ probe) {
    if (probe->select != (VEC256 ? 3 : 2)) return;
    using Mo = Moments<K>;
    constexpr int NB = Mo::NB, NY = Mo::NY, NS = NB + NY;      // sums per lane
    constexpr int kWarps = kRasterWarps;
    extern __shared__ __align__(16) unsigned char raster_smem[];
    // per warp: [32][NS] dim-2 sums of the run being flushed, then [32][NS] dim-1 factors beta_p(t1), gamma_p(t1)
    double (*s_S)[32][NS] = reinterpret_cast<double (*)[32][NS]>(raster_smem);
    double (*s_B)[32][NS] = reinterpret_cast<double (*)[32][NS]>(raster_smem + sizeof(double) * kWarps * 32 * NS);
    const Mesh mesh1 = load_mesh2(knots1, nk1), mesh2 = load_mesh2(knots2, nk2);
    const int nc2 = nk2 - 1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t n2 = probe->n2, n1 = n / n2;
    double (*S)[NS] = s_S[warp];
    double (*Bf)[NS] = s_B[warp];

    // tasks: 32-row groups x column segments (multiples of 4 columns), dealt round-robin to the warps of the grid
    const int64_t n_groups = (n1 + 31) / 32;
    const int64_t total_warps = (int64_t)gridDim.x * kWarps;
    int64_t n_seg = (4 * total_warps + n_groups - 1) / n_groups;           // ~4 tasks per warp
    int64_t seg_len = ((n2 + n_seg - 1) / n_seg + 3) & ~(int64_t)3;
    if (seg_len < 64) seg_len = 64;
    n_seg = (n2 + seg_len - 1) / seg_len;
    const int64_t n_tasks = n_groups * n_seg;

    double s[NB], sy[NY];
    double yy = 0.0;

    for (int64_t task = (int64_t)blockIdx.x * kWarps + warp; task < n_tasks; task += total_warps) {
        const int64_t g = task / n_seg, sg = task % n_seg;
        const int64_t row = g * 32 + lane;
        const bool active = row < n1;
        const int64_t c_begin = sg * seg_len, c_end = c_begin + seg_len < n2 ? c_begin + seg_len : n2;
        const TX* xr = X + 2 * (row * n2);
        const TY* yr = y + row * n2;
#pragma unroll
        for (int i = 0; i < NB; ++i) s[i] = 0.0;
#pragma unroll
        for (int i = 0; i < NY; ++i) sy[i] = 0.0;
        long long cur_x1 = 0;
        bool have_x1 = false, dirty = false;
        Interval i1, i2;
        i1.reset(); i2.reset();

        // warp-cooperative flush of every lane's current sums
        auto flush_all = [&]() {
#pragma unroll
            for (int q = 0; q < NB; ++q) S[lane][q] = s[q];
#pragma unroll
            for (int q = 0; q < NY; ++q) S[lane][NB + q] = sy[q];
            const int cell = dirty ? i1.idx * nc2 + i2.idx : -1;
            __syncwarp();
            unsigned remaining = __ballot_sync(0xffffffffu, cell >= 0);
            while (remaining) {
                const int leader = __ffs(remaining) - 1;
                const int cl = __shfl_sync(0xffffffffu, cell, leader);
                const unsigned grp = __ballot_sync(0xffffffffu, cell == cl) & remaining;
                double* dst = cellmom + (int64_t)cl * Mo::kAll;
                for (int o = lane; o < Mo::kAll; o += 32) {
                    const int pi = o < Mo::kGram ? o / NB : NB + (o - Mo::kGram) / NY;
                    const int qi = o < Mo::kGram ? o % NB : NB + (o - Mo::kGram) % NY;
                    double acc = 0.0;
                    unsigned m = grp;
                    while (m) {
                        const int e = __ffs(m) - 1;
                        m &= m - 1;
                        acc = fma(Bf[e][pi], S[e][qi], acc);
                    }
                    atomicAdd(dst + o, acc);
                }
                remaining &= ~grp;
            }
            __syncwarp();
#pragma unroll
            for (int q = 0; q < NB; ++q) s[q] = 0.0;
#pragma unroll
            for (int q = 0; q < NY; ++q) sy[q] = 0.0;
            dirty = false;
        };
        auto add = [&](double x1, double x2, double yv, bool valid) {
            const long long bits = __double_as_longlong(x1);
            const bool same_x1 = have_x1 && bits == cur_x1;
            const bool need = valid && !(same_x1 && i2.inside(x2));
            if (__any_sync(0xffffffffu, need)) {
                flush_all();
                if (need) {
                    if (!same_x1) {
                        if (!i1.inside(x1)) i1.set(mesh1, locate_interval(mesh1, x1, LdgLoader2()));
                        const double t1 = (x1 - i1.u) * mesh1.inv_delta;
                        double tp[2 * K + 1], up[2 * K + 1];
                        powers<2 * K>(t1, tp, up);
#pragma unroll
                        for (int p = 0; p < NB; ++p) Bf[lane][p] = tp[p] * up[2 * K - p];
#pragma unroll
                        for (int p = 0; p < NY; ++p) Bf[lane][NB + p] = tp[p] * up[K - p];
                        cur_x1 = bits;
                        have_x1 = true;
                    }
                    if (!i2.inside(x2)) i2.set(mesh2, locate_interval(mesh2, x2, LdgLoader2()));
                }
            }
            if (valid) {
                const double t2 = (x2 - i2.u) * mesh2.inv_delta;
                double tp[2 * K + 1], up[2 * K + 1];
                powers<2 * K>(t2, tp, up);
#pragma unroll
                for (int q = 0; q < NB; ++q) s[q] += tp[q] * up[2 * K - q];
#pragma unroll
                for (int q = 0; q < NY; ++q) sy[q] = fma(yv, tp[q] * up[K - q], sy[q]);
                yy = fma(yv, yv, yy);
                dirty = true;
            }
        };

        if (VEC256) {
            // n2 % 4 == 0 and 32-byte aligned bases: four points = two 256-bit loads of X and one of y (float32: 128-bit
            // loads), the next group's loads in flight while the current one is processed
            double xa[4], xb[4], ya[4];
            int64_t c = c_begin;
            if (active && c < c_end) { ldg4(xr + 2 * c, xa); ldg4(xr + 2 * c + 4, xb); ldg4(yr + c, ya); }
            for (; c < c_end; c += 4) {
                double ca[4], cb[4], cy[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) { ca[i] = xa[i]; cb[i] = xb[i]; cy[i] = ya[i]; }
                if (active && c + 4 < c_end) { ldg4(xr + 2 * (c + 4), xa); ldg4(xr + 2 * (c + 4) + 4, xb); ldg4(yr + c + 4, ya); }
                add(ca[0], ca[1], cy[0], active);
                add(ca[2], ca[3], cy[1], active);
                add(cb[0], cb[1], cy[2], active);
                add(cb[2], cb[3], cy[3], active);
            }
        } else {
            double2 pn = make_double2(0.0, 0.0);
            double yn = 0.0;
            if (active && c_begin < c_end) { pn = ldg_point(xr, c_begin); yn = ldg_d(yr + c_begin); }
            for (int64_t c = c_begin; c < c_end; ++c) {
                const double2 pc = pn;
                const double yc = yn;
                if (active && c + 1 < c_end) { pn = ldg_point(xr, c + 1); yn = ldg_d(yr + c + 1); }
                add(pc.x, pc.y, yc, active);
            }
        }
        flush_all();
    }

    __shared__ double s_yy[kWarps];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) yy += __shfl_xor_sync(0xffffffffu, yy, o);
    if (lane == 0) s_yy[warp] = yy;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int w = 0; w < kWarps; ++w) tot += s_yy[w];
        atomicAdd(scal, tot);
        if (blockIdx.x == 0) atomicAdd(scal + 1, (double)n);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// "column sweep" path: the raster is separable as well (every row carries the same x2 values, as np.meshgrid /
// lon-lat grids do).  The lanes of a warp take 32 CONSECUTIVE COLUMNS and sweep down the rows, so every load is a
// fully coalesced 512-byte (X) / 256-byte (y) request like in the 1-D kernel, each lane's x2 — hence its dim-2
// factors — never changes, the dim-1 sums are accumulated per lane, and all lanes cross a knot of dimension 1 at the
// same step (x1 is shared by the whole row), so the flush is again convergent and cooperative.  Roles of the two
// dimensions are swapped with respect to the row-streaming kernel above; the same per-lane checks keep any input
// correct.
// ------------------------------------------------------------------------------------------------------------------
// Warp-cooperative flush of the column-sweep kernel, out of line (it runs once per ~n1/(m1-k) rows).  Every lane has
// put its own dim-1 sums in S[lane][*] (Gram part: only what the row-by-row path added; projection part: everything)
// and the warp-uniform Gram sums in SU[*]; Bf[lane][*] are the lanes' dim-2 factors.  Lanes are grouped by cell; for a
// group g the Gram moments are  SU[p] * sum_{e in g} Bf[e][q]  (+ sum_e S[e][p] Bf[e][q] if `per_lane_gram`), the
// projection moments  sum_e S[e][NB+p] Bf[e][NB+q]; they leave as a few fp64 REDs per lane.
template <int K>
__device__ __noinline__ void flush_cols_2d(const double* __restrict__ S, const double* __restrict__ SU,
                                           const double* __restrict__ Bf, double* __restrict__ GB, int cell,
                                           bool per_lane_gram, double* __restrict__ cellmom) {
    using Mo = Moments<K>;
    constexpr int NB = Mo::NB, NY = Mo::NY, NS = NB + NY;
    const int lane = threadIdx.x & 31;
    __syncwarp();
    unsigned remaining = __ballot_sync(0xffffffffu, cell >= 0);
    while (remaining) {
        const int leader = __ffs(remaining) - 1;
        const int cl = __shfl_sync(0xffffffffu, cell, leader);
        const unsigned grp = __ballot_sync(0xffffffffu, cell == cl) & remaining;
        const int e_lo = __ffs(grp) - 1, e_hi = 31 - __clz(grp);
        double* dst = cellmom + (int64_t)cl * Mo::kAll;
        // GB[q] = sum over the group of the dim-2 Gram factors (lanes 0..NB-1, one q each).  The sums over the group's lanes
        // below run on four independent accumulators: a single FMA chain over up to 32 lanes was a fifth of the sweep's time.
        auto in_grp = [&](int e) { return e <= e_hi && ((grp >> e) & 1u); };
        if (lane < NB) {
            double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
            for (int e = e_lo; e <= e_hi; e += 4) {
                a0 += Bf[e * NS + lane];                                  // e_lo itself is in the group
                if (in_grp(e + 1)) a1 += Bf[(e + 1) * NS + lane];
                if (in_grp(e + 2)) a2 += Bf[(e + 2) * NS + lane];
                if (in_grp(e + 3)) a3 += Bf[(e + 3) * NS + lane];
            }
            GB[lane] = (a0 + a1) + (a2 + a3);
        }
        __syncwarp();
        for (int o = lane; o < Mo::kGram; o += 32) {
            const int pi = o / NB, qi = o % NB;
            double acc = SU[pi] * GB[qi];
            if (per_lane_gram) {
                for (int e = e_lo; e <= e_hi; ++e)
                    if ((grp >> e) & 1u) acc = fma(S[e * NS + pi], Bf[e * NS + qi], acc);
            }
            atomicAdd(dst + o, acc);
        }
        for (int o = lane; o < Mo::kProj; o += 32) {
            const int pi = NB + o / NY, qi = NB + o % NY;
            double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
            for (int e = e_lo; e <= e_hi; e += 4) {
                if (in_grp(e)) a0 = fma(S[e * NS + pi], Bf[e * NS + qi], a0);
                if (in_grp(e + 1)) a1 = fma(S[(e + 1) * NS + pi], Bf[(e + 1) * NS + qi], a1);
                if (in_grp(e + 2)) a2 = fma(S[(e + 2) * NS + pi], Bf[(e + 2) * NS + qi], a2);
                if (in_grp(e + 3)) a3 = fma(S[(e + 3) * NS + pi], Bf[(e + 3) * NS + qi], a3);
            }
            atomicAdd(dst + Mo::kGram + o, (a0 + a1) + (a2 + a3));
        }
        __syncwarp();
        remaining &= ~grp;
    }
    __syncwarp();
}

// A point whose x1 is not its row's x1 (the input is not the raster the probe took it for): added on its own, straight
// to the moment table.  Kept out of line so that it costs the sweep no registers.
template <int K>
__device__ __noinline__ void scatter_point_2d(const Mesh mesh1, const Mesh mesh2, double x1, double x2, double yv,
                                              double* __restrict__ cellmom) {
    using Mo = Moments<K>;
    constexpr int NB = Mo::NB, NY = Mo::NY;
    const int c1 = locate_interval(mesh1, x1, LdgLoader2()), c2 = locate_interval(mesh2, x2, LdgLoader2());
    double tp1[2 * K + 1], up1[2 * K + 1], tp2[2 * K + 1], up2[2 * K + 1];
    powers<2 * K>((x1 - __ldg(mesh1.knots + c1)) * mesh1.inv_delta, tp1, up1);
    powers<2 * K>((x2 - __ldg(mesh2.knots + c2)) * mesh2.inv_delta, tp2, up2);
    double* dst = cellmom + ((int64_t)c1 * (mesh2.n_knots - 1) + c2) * Mo::kAll;
#pragma unroll 1
    for (int p = 0; p < NB; ++p)
#pragma unroll 1
        for (int q = 0; q < NB; ++q) atomicAdd(dst + p * NB + q, tp1[p] * up1[2 * K - p] * tp2[q] * up2[2 * K - q]);
#pragma unroll 1
    for (int p = 0; p < NY; ++p)
#pragma unroll 1
        for (int q = 0; q < NY; ++q) atomicAdd(dst + Mo::kGram + p * NY + q, yv * tp1[p] * up1[K - p] * tp2[q] * up2[K - q]);
}

// Measured: the sweep runs at (bytes in flight) / (loaded DRAM latency, ~2 us) — with one group of four rows staged in
// registers (3 KB per warp, 48 KB per SM) it sits at 3.3 TB/s whatever the instruction count.  So the column walk is
// staged through shared memory instead: every lane cp.async's its own 16 B of X and 8 B of y, kColsRing rows deep
// (18 KB per warp, ~140 KB per SM in flight, no registers, no cross-lane synchronisation because a lane only ever reads
// what it copied itself).  Tried and measured slower (r02): the same ring filled by tiled TMA loads — one 4 x 512 B box of X
// and one 4 x 256 B box of y per group of four rows, issued by one lane, completion on a per-group mbarrier — 0.640 ms
// against 0.578 ms, with the barrier probe issued a group ahead; the 80 instructions of per-lane address arithmetic it
// removes were not on the critical path (stall_wait/short_sb dominate, two warps per scheduler), and such small boxes do
// not suit the TMA engine.
constexpr int kColsWarps = 8;
template <int K> struct ColsRing {       // rows in the ring: what fits beside the (K-dependent) tables in 227 KB
    static constexpr int kRows = K <= 3 ? 24 : (K == 4 ? 20 : (K == 5 ? 16 : 12));   // K = 6 at 16 rows exceeded 227 KB with the static arrays
};

__device__ __forceinline__ void cp_async_16(void* dst_smem, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_8(void* dst_smem, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
template <int BYTES> __device__ __forceinline__ void cp_async_stream(unsigned dst_smem, const void* src, uint64_t pol) {
    static_assert(BYTES == 16 || BYTES == 8 || BYTES == 4, "cp.async copies 4, 8 or 16 bytes");
    if constexpr (BYTES == 16) cp_async_16_stream(dst_smem, src, pol);
    else if constexpr (BYTES == 8) cp_async_8_stream(dst_smem, src, pol);
    else cp_async_4_stream(dst_smem, src, pol);
}
// one point (x1, x2) in the element type of X: the column sweep's ring holds the points as they are stored
template <class T> struct Pair;
template <> struct Pair<double> { using type = double2; };
template <> struct Pair<float> { using type = float2; };
__device__ __forceinline__ double2 to_double2(const double2 p) { return p; }
__device__ __forceinline__ double2 to_double2(const float2 p) { return make_double2(p.x, p.y); }
template <int K, class TX, class TY>
constexpr size_t cols_smem() {
    return sizeof(double) * 3 * kColsWarps * 32 * (3 * (size_t)K + 2)                                   // sums, factors, per-row table
           + (size_t)kColsWarps * ColsRing<K>::kRows * 32 * (sizeof(typename Pair<TX>::type) + sizeof(TY));   // the ring
}

template <int K, class TX, class TY>
__global__ void __launch_bounds__(kColsWarps * 32, 1)
accum_2d_cols_kernel(const TX* __restrict__ X, const TY* __restrict__ y, int64_t n,
                     const double* __restrict__ knots1, int nk1, const double* __restrict__ knots2, int nk2,
                     double* __restrict__ cellmom, double* __restrict__ scal, const ProbeResult* __restrict__ probe,
                     int hint_n2, int tasks_per_warp) {
    // hint_n2 > 0: the caller states that the input is a flattened raster with rows of hint_n2 points (asvgp_accum_2d_raster);
    // no probe ran.  The per-point checks below make a wrong statement slow, never wrong.
    if (hint_n2 <= 0 && probe->select != 4) return;
    using Mo = Moments<K>;
    constexpr int NB = Mo::NB, NY = Mo::NY, NS = NB + NY;
    constexpr int kWarps = kColsWarps;
    constexpr int kColsRing = ColsRing<K>::kRows;
    extern __shared__ __align__(16) unsigned char raster_smem[];
    // per warp: [32][NS] per-lane dim-1 sums being flushed | [32][NS] per-lane dim-2 factors | [32][NS] dim-1 factors of
    // the next 32 rows (x1 is shared by a whole row, so they are computed once per row, not once per point)
    double (*s_S)[32][NS] = reinterpret_cast<double (*)[32][NS]>(raster_smem);
    double (*s_B)[32][NS] = reinterpret_cast<double (*)[32][NS]>(raster_smem + sizeof(double) * kWarps * 32 * NS);
    double (*s_T)[32][NS] = reinterpret_cast<double (*)[32][NS]>(raster_smem + 2 * sizeof(double) * kWarps * 32 * NS);
    // per warp: ring of kColsRing rows, [row][lane] point of X then [row][lane] y, in their element types
    using PX = typename Pair<TX>::type;
    unsigned char* ring_base = raster_smem + 3 * sizeof(double) * kWarps * 32 * NS;
    PX* ringX = reinterpret_cast<PX*>(ring_base) + (size_t)(threadIdx.x >> 5) * kColsRing * 32;
    TY* ringY = reinterpret_cast<TY*>(ring_base + sizeof(PX) * kWarps * kColsRing * 32) + (size_t)(threadIdx.x >> 5) * kColsRing * 32;
    __shared__ __align__(16) long long s_bits[kWarps][32];     // x1 bit pattern of each table row
    __shared__ __align__(16) int s_cell[kWarps][32];           // its knot interval
    // per group of four table rows: sum over the rows of the Gram factors beta_p(t1) (the same for every column, so on a
    // separable raster the Gram moments need no per-point work at all), and the group's interval (-1: rows of the group
    // lie in different intervals or do not all exist -> row-by-row path)
    __shared__ __align__(16) double s_gsum[kWarps][8][NB + 1];
    __shared__ int s_gcell[kWarps][8];
    __shared__ double s_su[kWarps][NB], s_gb[kWarps][NB];      // flush: warp-uniform Gram sums, per-group factor sums
    // the dim-1 knots in shared memory: every 32-row block looks its rows' intervals up again (a lane's rows are 32 apart), and
    // the three dependent knot loads of a lookup cost 7 % of the sweep when they go to L1/L2 (ncu, r02)
    constexpr int kKnotsStaged = 512;
    __shared__ double s_knots1[kKnotsStaged];
    const Mesh mesh1 = load_mesh2(knots1, nk1), mesh2 = load_mesh2(knots2, nk2);
    Mesh mesh1s = mesh1;
    if (nk1 <= kKnotsStaged) {
        for (int i = threadIdx.x; i < nk1; i += blockDim.x) s_knots1[i] = __ldg(knots1 + i);
        mesh1s.knots = s_knots1;
    }
    __syncthreads();
    const int nc2 = nk2 - 1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t n2 = hint_n2 > 0 ? hint_n2 : probe->n2, n1 = n / n2;
    double (*S)[NS] = s_S[warp];
    double (*Bf)[NS] = s_B[warp];
    double (*T)[NS] = s_T[warp];
    long long* Tbits = s_bits[warp];
    int* Tcell = s_cell[warp];
    double (*Gsum)[NB + 1] = s_gsum[warp];
    int* Gcell = s_gcell[warp];

    // tasks: 32-column strips x row segments, dealt round-robin to the warps of the grid
    const uint64_t stream_policy = evict_first_policy();      // the points are read once: the 20 MB moment table stays in L2
    const int64_t n_strips = (n2 + 31) / 32;
    const int64_t total_warps = (int64_t)gridDim.x * kWarps;
    int64_t n_seg = (tasks_per_warp * total_warps + n_strips - 1) / n_strips;
    int64_t seg_len = ((n1 + n_seg - 1) / n_seg + 31) & ~(int64_t)31;
    if (seg_len < 64) seg_len = 64;
    n_seg = (n1 + seg_len - 1) / seg_len;
    const int64_t n_tasks = n_strips * n_seg;
    const PX* __restrict__ X2 = reinterpret_cast<const PX*>(X);

    double s[NB], sy[NY];
    double su[NB];                       // warp-uniform part of the dim-1 Gram sums (fast path); a lane's sum is s + su
    double yy = 0.0;

    constexpr long long kNoX2 = 0x7ff8dead0000beefLL;      // a NaN payload no input coordinate carries

    for (int64_t task = (int64_t)blockIdx.x * kWarps + warp; task < n_tasks; task += total_warps) {
        // consecutive warps take ADJACENT strips of the same row segment: a CTA then reads 8 x 512 B contiguous bytes of every
        // row, which keeps DRAM pages open
        const int64_t sg = task / n_strips, strip = task % n_strips;
        const int64_t col = strip * 32 + lane;
        const bool active = col < n2;
        const int64_t colc = active ? col : n2 - 1;        // lanes past the last column shadow it; they never flush
        const int64_t r_begin = sg * seg_len, r_end = r_begin + seg_len < n1 ? r_begin + seg_len : n1;
#pragma unroll
        for (int i = 0; i < NB; ++i) { s[i] = 0.0; su[i] = 0.0; }
#pragma unroll
        for (int i = 0; i < NY; ++i) sy[i] = 0.0;
        long long cur_x2 = kNoX2;
        bool dirty = false;
        bool any_slow = false;           // warp-uniform: some lane's own Gram sums s[] are non-zero
        int cur_c1 = -1;                 // warp-uniform: dim-1 interval the lane sums belong to
        double yy_task = 0.0;
        Interval it, i2;                 // it: interval cache of the table builder
        it.reset(); i2.reset();

        auto flush_all = [&]() {
#pragma unroll
            for (int q = 0; q < NB; ++q) S[lane][q] = s[q];
#pragma unroll
            for (int q = 0; q < NY; ++q) S[lane][NB + q] = sy[q];
            if (lane == 0) {
#pragma unroll
                for (int q = 0; q < NB; ++q) s_su[warp][q] = su[q];
            }
            flush_cols_2d<K>(&S[0][0], s_su[warp], &Bf[0][0], s_gb[warp], (dirty && active) ? cur_c1 * nc2 + i2.idx : -1,
                             any_slow, cellmom);
            any_slow = false;
#pragma unroll
            for (int q = 0; q < NB; ++q) { s[q] = 0.0; su[q] = 0.0; }
#pragma unroll
            for (int q = 0; q < NY; ++q) sy[q] = 0.0;
            dirty = false;
        };
        // one point of table row `row`; everything here is warp-uniform except inside the `odd` branch
        auto process = [&](int row, const double2 pt, const double yv) {
            const int c1 = Tcell[row];
            if (c1 != cur_c1) {                                   // the row entered another dim-1 interval
                flush_all();
                cur_c1 = c1;
            }
            const long long bx = __double_as_longlong(pt.x), by = __double_as_longlong(pt.y);
            bool skip = false;
            if (__any_sync(0xffffffffu, ((bx ^ Tbits[row]) | (by ^ cur_x2)) != 0)) {
                flush_all();
                if (by != cur_x2) {                               // first point of the task, or x2 is not constant
                    if (!i2.inside(pt.y)) i2.set(mesh2, locate_interval(mesh2, pt.y, LdgLoader2()));
                    double tp[2 * K + 1], up[2 * K + 1];
                    powers<2 * K>((pt.y - i2.u) * mesh2.inv_delta, tp, up);
#pragma unroll
                    for (int q = 0; q < NB; ++q) Bf[lane][q] = tp[q] * up[2 * K - q];
#pragma unroll
                    for (int q = 0; q < NY; ++q) Bf[lane][NB + q] = tp[q] * up[K - q];
                    cur_x2 = by;
                }
                if (bx != Tbits[row]) {                           // not the raster the probe took it for
                    if (active) scatter_point_2d<K>(mesh1, mesh2, pt.x, pt.y, yv, cellmom);
                    skip = true;
                }
            }
            yy_task = fma(yv, yv, yy_task);
            any_slow = true;
            if (!skip) {
                const double* Tr = T[row];
#pragma unroll
                for (int p = 0; p < NB; ++p) s[p] += Tr[p];
#pragma unroll
                for (int p = 0; p < NY; ++p) sy[p] = fma(yv, Tr[NB + p], sy[p]);
                dirty = true;
            }
        };

        // ---- the column walk, pipelined kColsRing rows deep through the shared-memory ring -------------------------
        const int64_t rows_total = r_end - r_begin;
        const int64_t n_groups = (rows_total + 3) >> 2;               // groups of four rows (the last may be ragged)
        const PX* xq = X2 + r_begin * n2 + colc;                      // next row to request: += n2 per row
        const TY* yq = y + r_begin * n2 + colc;
        int to_request = (int)rows_total;                             // rows not requested yet (a segment is < 2^31 rows)
        int wslot = 0;                                                // ring slot of the next request (32-bit, no modulo)
        auto request_group = [&]() {                                  // one commit group = up to four rows
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (to_request > 0) {
                    cp_async_stream<sizeof(PX)>(smem_u32(ringX + wslot * 32 + lane), xq, stream_policy);
                    cp_async_stream<sizeof(TY)>(smem_u32(ringY + wslot * 32 + lane), yq, stream_policy);
                    xq += n2;
                    yq += n2;
                    --to_request;
                }
                wslot = wslot + 1 == kColsRing ? 0 : wslot + 1;       // slots advance in whole groups, rows or not
            }
            cp_async_commit();
        };
        constexpr int kGroupsInFlight = kColsRing / 4 - 1;            // one group's slots are being read
#pragma unroll
        for (int g = 0; g < kGroupsInFlight; ++g) request_group();
        int rslot = 0;                                                // ring slot of the next row to consume
        // x1 of table row `lane` of the next 32-row block, requested one block ahead so that its DRAM latency is hidden
        double x1_next = (r_begin + lane < r_end) ? ldg_d(X + 2 * ((r_begin + lane) * n2 + strip * 32)) : 0.0;

        for (int64_t r0 = r_begin; r0 < r_end; r0 += 32) {
            // ---- dim-1 factors of rows r0 .. r0+31: lane l does row r0 + l ---------------------------------------------
            __syncwarp();
            {
                const int64_t r = r0 + lane;
                const double x1 = x1_next;
                if (r + 32 < r_end) x1_next = ldg_d(X + 2 * ((r + 32) * n2 + strip * 32));
                if (r < r_end) {
                    if (!it.inside(x1)) it.set(mesh1s, locate_interval(mesh1s, x1, PlainLoader2()), PlainLoader2());
                    double tp[2 * K + 1], up[2 * K + 1];
                    powers<2 * K>((x1 - it.u) * mesh1.inv_delta, tp, up);
#pragma unroll
                    for (int p = 0; p < NB; ++p) T[lane][p] = tp[p] * up[2 * K - p];
#pragma unroll
                    for (int p = 0; p < NY; ++p) T[lane][NB + p] = tp[p] * up[K - p];
                    Tbits[lane] = __double_as_longlong(x1);
                    Tcell[lane] = it.idx;
                }
            }
            __syncwarp();
            const int n_rows = (int)(r_end - r0 < 32 ? r_end - r0 : 32);
            if (lane < 8) {                                      // lane g sums the factors of rows 4g .. 4g+3
                const int g4 = 4 * lane;
                int gc = -1;
                if (g4 + 3 < n_rows) {
                    gc = Tcell[g4];
                    if (Tcell[g4 + 1] != gc || Tcell[g4 + 2] != gc || Tcell[g4 + 3] != gc) gc = -1;
#pragma unroll
                    for (int p = 0; p < NB; ++p) Gsum[lane][p] = (T[g4][p] + T[g4 + 1][p]) + (T[g4 + 2][p] + T[g4 + 3][p]);
                }
                Gcell[lane] = gc;
            }
            __syncwarp();
            for (int u0 = 0; u0 < n_rows; u0 += 4) {
                // the oldest group has landed; read it, then hand its slots to a new request
                cp_async_wait<kGroupsInFlight - 1>();
                double2 cx[4];
                double cy[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    cx[u] = to_double2(ringX[(rslot + u) * 32 + lane]);   // groups never straddle the end of the ring
                    cy[u] = (double)ringY[(rslot + u) * 32 + lane];
                }
                rslot = rslot + 4 == kColsRing ? 0 : rslot + 4;
                request_group();
                if (u0 + 3 < n_rows) {
                    // fast path: the four rows lie in one interval and every lane sees its row's x1 and its own x2
                    const int gc = Gcell[u0 >> 2];
                    long long odd = 0;
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        odd |= (__double_as_longlong(cx[u].x) ^ Tbits[u0 + u]) | (__double_as_longlong(cx[u].y) ^ cur_x2);
                    if (gc >= 0 && !__any_sync(0xffffffffu, odd != 0)) {
                        if (gc != cur_c1) {
                            flush_all();
                            cur_c1 = gc;
                        }
                        const double* gs = Gsum[u0 >> 2];
#pragma unroll
                        for (int p = 0; p < NB; ++p) su[p] += gs[p];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const double* Tr = T[u0 + u] + NB;
#pragma unroll
                            for (int p = 0; p < NY; ++p) sy[p] = fma(cy[u], Tr[p], sy[p]);
                            yy_task = fma(cy[u], cy[u], yy_task);
                        }
                        dirty = true;
                    } else {
#pragma unroll
                        for (int u = 0; u < 4; ++u) process(u0 + u, cx[u], cy[u]);
                    }
                } else {
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (u0 + u < n_rows) process(u0 + u, cx[u], cy[u]);
                }
            }
        }
        cp_async_wait<0>();
        flush_all();
        if (active) yy += yy_task;
    }

    __shared__ double s_yy[kWarps];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) yy += __shfl_xor_sync(0xffffffffu, yy, o);
    if (lane == 0) s_yy[warp] = yy;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int w = 0; w < kWarps; ++w) tot += s_yy[w];
        atomicAdd(scal, tot);
        if (blockIdx.x == 0) atomicAdd(scal + 1, (double)n);
    }
}

// Probe (one CTA): classifies the input without a host round trip.
//   raster  : n2 = position of the first change of x1 (searched in the first 2^20 points) divides n, and at 1024 sampled
//             rows the first and last point share x1 while the previous row's last point does not
//   separable raster : additionally x2 of 1024 sampled points equals x2 of the same column in the first row
//   x1-run  : at least three quarters of 4096 sampled points share x1 with their successor
//   general : everything else
// (Bit patterns are compared on the values converted to double: the conversion from float is exact and one-to-one, so that
// is the comparison in the source type.)
template <class TX, class TY>
__global__ void __launch_bounds__(1024) accum_2d_probe_kernel(const TX* __restrict__ X, const TY* __restrict__ y,
                                                              int64_t n, ProbeResult* __restrict__ out) {
    // 1024 threads, every thread's samples issued back to back: the probe costs a handful of DRAM round trips
    __shared__ int s_cnt[32];
    __shared__ long long s_first;
    const int tid = threadIdx.x;
    auto x1bits = [&](int64_t i) { return __double_as_longlong(ldg_d(X + 2 * i)); };
    // fraction of points equal to their successor (4 samples per thread)
    const int n_probe = (int)(n - 1 < 4096 ? n - 1 : 4096);
    int hits = 0;
    {
        long long a[4], b[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = tid + u * 1024;
            const int64_t i = j < n_probe ? (int64_t)((double)j * (double)(n - 1) / (double)n_probe) : 0;
            a[u] = x1bits(i);
            b[u] = x1bits(i + (n > 1 ? 1 : 0));
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) hits += (tid + u * 1024 < n_probe) && a[u] == b[u];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) hits += __shfl_xor_sync(0xffffffffu, hits, o);
    if ((tid & 31) == 0) s_cnt[tid >> 5] = hits;
    if (tid == 0) s_first = -1;
    __syncthreads();
    int tot = 0;
    for (int w = 0; w < 32; ++w) tot += s_cnt[w];
    const bool runs = n_probe > 0 && 4 * tot >= 3 * n_probe;
    // first change of x1 (searched in the first 2^20 points, 8192 positions per round)
    const long long b0 = x1bits(0);
    const int64_t limit = n < (1 << 20) ? n : (1 << 20);
    for (int64_t base = 1; base < limit; base += 8 * 1024) {
        long long v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int64_t i = base + tid + (int64_t)u * 1024;
            v[u] = i < limit ? x1bits(i) : b0;
        }
        long long first = -1;
#pragma unroll
        for (int u = 7; u >= 0; --u)
            if (v[u] != b0) first = base + tid + (int64_t)u * 1024;
        if (first >= 0) atomicMin(reinterpret_cast<unsigned long long*>(&s_first), (unsigned long long)first);
        if (__syncthreads_or(first >= 0)) break;
    }
    __syncthreads();
    const long long n2 = s_first;             // -1 when no change was found
    bool raster = runs && n2 > 1 && n % n2 == 0;
    bool separable = false;
    if (raster) {                             // block-uniform
        const int64_t n1 = n / n2;
        // one sampled row per thread: first and last point share x1, the previous row's last point does not; and one
        // sampled point per thread carries the x2 of its column in the first row
        const int64_t r = (int64_t)((double)tid * (double)(n1 - 1) / 1023.0 + 0.5);
        const long long a = x1bits(r * n2), e = x1bits(r * n2 + n2 - 1), pz = r > 0 ? x1bits(r * n2 - 1) : ~a;
        const int64_t rs = n1 > 1 ? 1 + (int64_t)((double)tid * (double)(n1 - 2) / 1023.0 + 0.5) : 0;
        const int64_t c = (int64_t)(((unsigned long long)tid * 2654435761ull) % (unsigned long long)n2);
        const long long s0 = __double_as_longlong(ldg_d(X + 2 * c + 1));
        const long long s1 = rs < n1 ? __double_as_longlong(ldg_d(X + 2 * (rs * n2 + c) + 1)) : s0;
        raster = !__syncthreads_or(a != e || a == pz);
        separable = !__syncthreads_or(s0 != s1) && raster;
    }
    if (tid == 0) {
        const bool aligned = ((reinterpret_cast<uintptr_t>(X) | reinterpret_cast<uintptr_t>(y)) & 31u) == 0;
        out->select = raster ? (separable ? 4 : ((n2 % 4 == 0 && aligned) ? 3 : 2)) : (runs ? 1 : 0);
        out->n2 = raster ? (int)n2 : 0;
    }
}

// Expands the per-cell moments into the Gram stencil and the projection:
//   G[(c1+r1, c2+r2), (c1+s1, c2+s2)] += sum_pq C[r1][s1][p] C[r2][s2][q] mom[p][q]      (lower part only)
//   b[(c1+r1, c2+r2)]                 += sum_pq D[r1][p] D[r2][q] ymom[p][q]
// One CTA per cell; thread = one (r1, s1, r2, s2) combination (or one (r1, r2) for b).
// Stencil layout: Gs[e * M + j], e = d1 * (2k+1) + (d2 + k), d1 = i1 - j1 in [0, k], d2 = i2 - j2 in [-k, k],
// j = j1 * m2 + j2; stored for (d1 > 0) or (d1 == 0 and d2 >= 0).
template <int K>
__global__ void __launch_bounds__(256) expand_moments_2d_kernel(const double* __restrict__ cellmom,
                                                               const double* __restrict__ Cprod,
                                                               const double* __restrict__ Dy, int nc1, int nc2, int m2,
                                                               int64_t M, double* __restrict__ Gs,
                                                               double* __restrict__ b) {
    using Mo = Moments<K>;
    constexpr int NB = Mo::NB, NY = Mo::NY, K1 = K + 1;
    __shared__ double s_mom[Mo::kAll];
    __shared__ double s_C[K1 * K1 * NB];
    __shared__ double s_D[K1 * NY];
    __shared__ double s_inner[K1 * K1 * NB];
    for (int i = threadIdx.x; i < K1 * K1 * NB; i += blockDim.x) s_C[i] = Cprod[i];
    for (int i = threadIdx.x; i < K1 * NY; i += blockDim.x) s_D[i] = Dy[i];
    // persistent CTAs over the cells: one CTA per cell (38 809 launches of a few hundred instructions at 200 x 200) was bound
    // by CTA turnover, not by its arithmetic or its REDs
    for (int cell = blockIdx.x; cell < nc1 * nc2; cell += gridDim.x) {
        const int c1 = cell / nc2, c2 = cell % nc2;
        __syncthreads();                           // the previous cell's readers are done with s_mom / s_inner
        for (int i = threadIdx.x; i < Mo::kAll; i += blockDim.x) s_mom[i] = cellmom[(int64_t)cell * Mo::kAll + i];
        __syncthreads();
        // stage 1: inner[(r2, s2)][p] = sum_q C[r2][s2][q] mom[p][q] — shared by every (r1, s1)
        for (int o = threadIdx.x; o < K1 * K1 * NB; o += blockDim.x) {
            const int p = o % NB, rs2 = o / NB;
            double inner = 0.0;
#pragma unroll
            for (int q = 0; q < NB; ++q) inner = fma(s_C[rs2 * NB + q], s_mom[p * NB + q], inner);
            s_inner[o] = inner;
        }
        __syncthreads();
        for (int o = threadIdx.x; o < K1 * K1 * K1 * K1; o += blockDim.x) {
            const int s2 = o % K1, r2 = (o / K1) % K1, s1 = (o / (K1 * K1)) % K1, r1 = o / (K1 * K1 * K1);
            const int d1 = r1 - s1, d2 = r2 - s2;
            if (d1 < 0 || (d1 == 0 && d2 < 0)) continue;
            double v = 0.0;
#pragma unroll
            for (int p = 0; p < NB; ++p) v = fma(s_C[(r1 * K1 + s1) * NB + p], s_inner[(r2 * K1 + s2) * NB + p], v);
            const int e = d1 * (2 * K + 1) + (d2 + K);
            const int64_t j = (int64_t)(c1 + s1) * m2 + (c2 + s2);
            atomicAdd(Gs + (int64_t)e * M + j, v);
        }
        for (int o = threadIdx.x; o < K1 * K1; o += blockDim.x) {
            const int r2 = o % K1, r1 = o / K1;
            double v = 0.0;
#pragma unroll
            for (int p = 0; p < NY; ++p) {
                double inner = 0.0;
#pragma unroll
                for (int q = 0; q < NY; ++q) inner = fma(s_D[r2 * NY + q], s_mom[Mo::kGram + p * NY + q], inner);
                v = fma(s_D[r1 * NY + p], inner, v);
            }
            atomicAdd(b + (int64_t)(c1 + r1) * m2 + (c2 + r2), v);
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// predictor: mean = w^T alpha, var = v1 v2 + w^T Sigma_P w - (a^T S1 a)(b^T S2 b),  w = a (x) b
// (reference gpr.py:321-332).  Only the stencil entries of P^-1 and the bands of K1^-1, K2^-1 are needed.
//
// Inside one cell (c1, c2) both are bivariate polynomials in the local coordinates (t1, t2): the mean of degree k, the
// variance of degree 2k per dimension.  A first kernel (one CTA per cell) turns the posterior into that
// piecewise-polynomial form — (k+1)^2 + (2k+1)^2 monomial coefficients per cell plus the two univariate factors —
// and the streaming kernel then needs no gathers from the stencil at all.  Every thread walks a contiguous slice of the
// test points and keeps, for the (x1, cell) it is in, the mean/variance reduced to polynomials in t2 alone; on a
// gridded test set (x1 constant along a row, ~n2/(m2-k) consecutive points per cell) a point costs one Horner of
// degree k and one of degree 2k (~12 fp64 instructions), scattered points cost one (k+1)^2 + (2k+1)^2 contraction
// each.  32 B of traffic per point (X in, mean and var out).
// ------------------------------------------------------------------------------------------------------------------
template <int K> struct PredTable {
    static constexpr int NM = (K + 1) * (K + 1);          // mean coefficients  [p][q], p, q = 0..k
    static constexpr int NV = (2 * K + 1) * (2 * K + 1);  // variance coefficients [P][Q], P, Q = 0..2k
    static constexpr int kCell = NM + NV;
    static constexpr int NQ = 2 * K + 1;                  // univariate a^T S1 a / b^T S2 b per 1-D cell
};

template <int K>
__global__ void __launch_bounds__(256) predict_2d_table_kernel(int nc1, int nc2, int m1, int m2,
                                                              const double* __restrict__ alpha,
                                                              const double* __restrict__ SigP,
                                                              const double* __restrict__ S1,
                                                              const double* __restrict__ S2,
                                                              double* __restrict__ table) {
    using PT = PredTable<K>;
    constexpr int K1 = K + 1, NS = 2 * K + 1, W = K1 * K1;
    __shared__ double s_A[K1][K1];               // A[r][p]
    __shared__ double s_AA[K1][K1][NS];          // AA[r][s][P]
    extern __shared__ __align__(16) double s_win[];   // [W][W] window of Sigma_P, then alpha window [W]
    double* s_alpha = s_win + W * W;
    const int64_t M = (int64_t)m1 * m2;
    const int tid = threadIdx.x;
    for (int i = tid; i < K1 * K1; i += blockDim.x) s_A[i / K1][i % K1] = 0.0;
    __syncthreads();
    if (tid < K1 * K1) {
        constexpr PieceTable<K> tab = make_piece_table<K>();
        const int r = tid / K1, p = tid % K1;
        s_A[r][p] = (double)tab.c[r][p] / (double)tab.fact;
    }
    for (int i = tid; i < K1 * K1 * NS; i += blockDim.x) {
        constexpr PieceTable<K> tab = make_piece_table<K>();
        const int P = i % NS, sidx = (i / NS) % K1, r = i / (NS * K1);
        long long acc = 0;
        for (int p = 0; p <= K; ++p) {
            const int pp = P - p;
            if (pp >= 0 && pp <= K) acc += tab.c[r][p] * tab.c[sidx][pp];
        }
        s_AA[r][sidx][P] = (double)acc / ((double)tab.fact * (double)tab.fact);
    }
    const int n_cells = nc1 * nc2;
    if ((int)blockIdx.x < n_cells) {
        const int c1 = blockIdx.x / nc2, c2 = blockIdx.x % nc2;
        // window of the symmetric Sigma_P: rows/cols (r1, r2) -> basis index (c1 + r1, c2 + r2)
        for (int i = tid; i < W * W; i += blockDim.x) {
            const int a = i / W, b = i % W;
            const int r1 = a / K1, r2 = a % K1, s1 = b / K1, s2 = b % K1;
            int d1 = r1 - s1, d2 = r2 - s2;
            int j1 = c1 + s1, j2 = c2 + s2;
            if (d1 < 0 || (d1 == 0 && d2 < 0)) { d1 = -d1; d2 = -d2; j1 = c1 + r1; j2 = c2 + r2; }
            s_win[i] = __ldg(SigP + (int64_t)(d1 * NS + d2 + K) * M + (int64_t)j1 * m2 + j2);
        }
        for (int i = tid; i < W; i += blockDim.x) s_alpha[i] = __ldg(alpha + (int64_t)(c1 + i / K1) * m2 + (c2 + i % K1));
        __syncthreads();
        double* out = table + (int64_t)blockIdx.x * PT::kCell;
        for (int o = tid; o < PT::NM; o += blockDim.x) {
            const int p = o / K1, q = o % K1;
            double v = 0.0;
            for (int r1 = 0; r1 < K1; ++r1) {
                double inner = 0.0;
                for (int r2 = 0; r2 < K1; ++r2) inner = fma(s_A[r2][q], s_alpha[r1 * K1 + r2], inner);
                v = fma(s_A[r1][p], inner, v);
            }
            out[o] = v;
        }
        // variance coefficients in two stages: contract dimension 2 first,
        //   U[(r1,s1)][Q] = sum_{r2,s2} AA[r2][s2][Q] Sigma[(r1,r2),(s1,s2)],   then   Cv[P][Q] = sum_{r1,s1} AA[r1][s1][P] U[(r1,s1)][Q]
        double* s_U = s_alpha + W;                       // [K1*K1][NS]
        for (int o = tid; o < K1 * K1 * NS; o += blockDim.x) {
            const int Q = o % NS, s1 = (o / NS) % K1, r1 = o / (NS * K1);
            double v = 0.0;
            for (int r2 = 0; r2 < K1; ++r2)
                for (int s2 = 0; s2 < K1; ++s2)
                    v = fma(s_AA[r2][s2][Q], s_win[(r1 * K1 + r2) * W + s1 * K1 + s2], v);
            s_U[o] = v;
        }
        __syncthreads();
        for (int o = tid; o < PT::NV; o += blockDim.x) {
            const int P = o / NS, Q = o % NS;
            double v = 0.0;
            for (int r1 = 0; r1 < K1; ++r1)
                for (int s1 = 0; s1 < K1; ++s1) v = fma(s_AA[r1][s1][P], s_U[(r1 * K1 + s1) * NS + Q], v);
            out[PT::NM + o] = v;
        }
    } else {
        // the two univariate factors: Q1[c][P] = sum_rs S1[c+r, c+s] AA[r][s][P] (and the same for dimension 2)
        __syncthreads();
        const int which = blockIdx.x - n_cells;          // 0: dimension 1, 1: dimension 2
        const int nc = which == 0 ? nc1 : nc2, m = which == 0 ? m1 : m2;
        const double* Sb = which == 0 ? S1 : S2;
        double* out = table + (int64_t)n_cells * PT::kCell + (which == 0 ? 0 : (int64_t)nc1 * PT::NQ);
        for (int o = tid; o < nc * PT::NQ; o += blockDim.x) {
            const int c = o / PT::NQ, P = o % PT::NQ;
            double v = 0.0;
            for (int r = 0; r < K1; ++r)
                for (int sidx = 0; sidx < K1; ++sidx) {
                    const int d = r - sidx;
                    const double sv = d >= 0 ? __ldg(Sb + (int64_t)d * m + c + sidx) : __ldg(Sb + (int64_t)(-d) * m + c + r);
                    v = fma(s_AA[r][sidx][P], sv, v);
                }
            out[o] = v;
        }
    }
}

__device__ __forceinline__ void stg256(double* p, const double (&v)[4]) {
    asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(v[0]), "d"(v[1]), "d"(v[2]), "d"(v[3]) : "memory");
}

template <int K, bool VEC256>
__global__ void __launch_bounds__(256, 2) predict_2d_kernel(const double* __restrict__ X, int64_t n,
                                                            const double* __restrict__ knots1, int nk1,
                                                            const double* __restrict__ knots2, int nk2,
                                                            const double* __restrict__ table, double prior_var,
                                                            double* __restrict__ mean, double* __restrict__ var,
                                                            const ProbeResult* __restrict__ probe) {
    if (probe->select == 4) return;                  // the column sweep handles separable rasters
    using PT = PredTable<K>;
    constexpr int K1 = K + 1, NS = 2 * K + 1;
    const Mesh mesh1 = load_mesh2(knots1, nk1), mesh2 = load_mesh2(knots2, nk2);
    const int nc1 = nk1 - 1, nc2 = nk2 - 1;
    const double* Q1 = table + (int64_t)nc1 * nc2 * PT::kCell;
    const double* Q2 = Q1 + (int64_t)nc1 * PT::NQ;

    const int64_t n_threads = (int64_t)gridDim.x * blockDim.x;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t per = (n + n_threads - 1) / n_threads;
    per = (per + 3) & ~(int64_t)3;
    const int64_t begin = tid * per < n ? tid * per : n;
    const int64_t end = begin + per < n ? begin + per : n;

    double mc[K1], vc[NS];               // mean / variance as polynomials in t2 for the current (x1, cell)
    double tp1[NS];                      // powers of t1 of the current x1
    double q1 = 0.0;
    long long cur_x1 = 0;
    bool have_x1 = false;
    Interval i1, i2;
    i1.reset(); i2.reset();

    auto eval = [&](double x1, double x2, double& mu, double& vv) {
        const long long bits = __double_as_longlong(x1);
        const bool same_x1 = have_x1 && bits == cur_x1;
        if (!(same_x1 && i2.inside(x2))) {
            if (!same_x1) {
                if (!i1.inside(x1)) i1.set(mesh1, locate_interval(mesh1, x1, LdgLoader2()));
                const double t1 = (x1 - i1.u) * mesh1.inv_delta;
                tp1[0] = 1.0;
#pragma unroll
                for (int i = 1; i < NS; ++i) tp1[i] = tp1[i - 1] * t1;
                q1 = 0.0;
#pragma unroll
                for (int P = NS - 1; P >= 0; --P) q1 = fma(q1, t1, __ldg(Q1 + (int64_t)i1.idx * PT::NQ + P));
                cur_x1 = bits;
                have_x1 = true;
            }
            if (!i2.inside(x2)) i2.set(mesh2, locate_interval(mesh2, x2, LdgLoader2()));
            const double* cell = table + ((int64_t)i1.idx * nc2 + i2.idx) * PT::kCell;
#pragma unroll
            for (int q = 0; q < K1; ++q) {
                double v = 0.0;
#pragma unroll
                for (int p = 0; p < K1; ++p) v = fma(__ldg(cell + p * K1 + q), tp1[p], v);
                mc[q] = v;
            }
#pragma unroll
            for (int Q = 0; Q < NS; ++Q) {
                double v = 0.0;
#pragma unroll
                for (int P = 0; P < NS; ++P) v = fma(__ldg(cell + PT::NM + P * NS + Q), tp1[P], v);
                vc[Q] = fma(-q1, __ldg(Q2 + (int64_t)i2.idx * PT::NQ + Q), v);
            }
            vc[0] += prior_var;
        }
        const double t2 = (x2 - i2.u) * mesh2.inv_delta;
        double m = mc[K];
#pragma unroll
        for (int q = K - 1; q >= 0; --q) m = fma(m, t2, mc[q]);
        double v = vc[2 * K];
#pragma unroll
        for (int Q = 2 * K - 1; Q >= 0; --Q) v = fma(v, t2, vc[Q]);
        mu = m;
        vv = v;
    };

    int64_t i = begin;
    if (VEC256) {
        const int64_t n_full = begin + ((end - begin) & ~(int64_t)3);
        double xa[4], xb[4];
        if (i < n_full) { ldg256(X + 2 * i, xa); ldg256(X + 2 * i + 4, xb); }
        for (; i < n_full; i += 4) {
            double ca[4], cb[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) { ca[j] = xa[j]; cb[j] = xb[j]; }
            if (i + 4 < n_full) { ldg256(X + 2 * (i + 4), xa); ldg256(X + 2 * (i + 4) + 4, xb); }
            double mu[4], vv[4];
            eval(ca[0], ca[1], mu[0], vv[0]);
            eval(ca[2], ca[3], mu[1], vv[1]);
            eval(cb[0], cb[1], mu[2], vv[2]);
            eval(cb[2], cb[3], mu[3], vv[3]);
            stg256(mean + i, mu);
            stg256(var + i, vv);
        }
    }
    const double2* __restrict__ X2 = reinterpret_cast<const double2*>(X);
    for (; i < end; ++i) {
        const double2 pt = __ldg(X2 + i);
        double mu, vv;
        eval(pt.x, pt.y, mu, vv);
        mean[i] = mu;
        var[i] = vv;
    }
}

// Column-sweep predictor for separable raster test sets (same classification probe as the accumulate): the lanes of a
// warp take 32 consecutive columns and walk down the rows, so loads (512 B) and stores (2 x 256 B) are coalesced; a
// lane's x2 never changes, so mean and variance are cached as polynomials in t1 for the (x2, dim-1 interval) the lane
// is in and a point costs two Horner evaluations.
template <int K>
__global__ void __launch_bounds__(256, 2) predict_2d_cols_kernel(const double* __restrict__ X, int64_t n,
                                                                 const double* __restrict__ knots1, int nk1,
                                                                 const double* __restrict__ knots2, int nk2,
                                                                 const double* __restrict__ table, double prior_var,
                                                                 double* __restrict__ mean, double* __restrict__ var,
                                                                 const ProbeResult* __restrict__ probe, int hint_n2) {
    if (hint_n2 <= 0 && probe->select != 4) return;
    using PT = PredTable<K>;
    constexpr int K1 = K + 1, NS = 2 * K + 1;
    const Mesh mesh1 = load_mesh2(knots1, nk1), mesh2 = load_mesh2(knots2, nk2);
    const int nc1 = nk1 - 1, nc2 = nk2 - 1;
    const double* Q1 = table + (int64_t)nc1 * nc2 * PT::kCell;
    const double* Q2 = Q1 + (int64_t)nc1 * PT::NQ;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t n2 = hint_n2 > 0 ? hint_n2 : probe->n2, n1 = n / n2;
    const int64_t n_strips = (n2 + 31) / 32;
    const int64_t total_warps = (int64_t)gridDim.x * 8;
    int64_t n_seg = (4 * total_warps + n_strips - 1) / n_strips;
    int64_t seg_len = ((n1 + n_seg - 1) / n_seg + 3) & ~(int64_t)3;
    if (seg_len < 64) seg_len = 64;
    n_seg = (n1 + seg_len - 1) / seg_len;
    const int64_t n_tasks = n_strips * n_seg;
    const double2* __restrict__ X2 = reinterpret_cast<const double2*>(X);
    constexpr long long kNoX2 = 0x7ff8dead0000beefLL;

    for (int64_t task = (int64_t)blockIdx.x * 8 + warp; task < n_tasks; task += total_warps) {
        const int64_t sg = task / n_strips, strip = task % n_strips;
        const int64_t col = strip * 32 + lane;
        if (col >= n2) continue;                       // no warp-level cooperation in this kernel
        const int64_t r_begin = sg * seg_len, r_end = r_begin + seg_len < n1 ? r_begin + seg_len : n1;
        double mc[K1], vc[NS], tp2[NS];
        double q2 = 0.0;
        long long cur_x2 = kNoX2;
        Interval i1, i2;
        i1.reset(); i2.reset();

        auto eval = [&](const double2 pt, double& mu, double& vv) {
            const long long by = __double_as_longlong(pt.y);
            if (by != cur_x2 || !i1.inside(pt.x)) {
                if (by != cur_x2) {
                    if (!i2.inside(pt.y)) i2.set(mesh2, locate_interval(mesh2, pt.y, LdgLoader2()));
                    const double t2 = (pt.y - i2.u) * mesh2.inv_delta;
                    tp2[0] = 1.0;
#pragma unroll
                    for (int i = 1; i < NS; ++i) tp2[i] = tp2[i - 1] * t2;
                    q2 = 0.0;
#pragma unroll
                    for (int Q = NS - 1; Q >= 0; --Q) q2 = fma(q2, t2, __ldg(Q2 + (int64_t)i2.idx * PT::NQ + Q));
                    cur_x2 = by;
                }
                if (!i1.inside(pt.x)) i1.set(mesh1, locate_interval(mesh1, pt.x, LdgLoader2()));
                const double* cell = table + ((int64_t)i1.idx * nc2 + i2.idx) * PT::kCell;
#pragma unroll
                for (int p = 0; p < K1; ++p) {
                    double v = 0.0;
#pragma unroll
                    for (int q = 0; q < K1; ++q) v = fma(__ldg(cell + p * K1 + q), tp2[q], v);
                    mc[p] = v;
                }
#pragma unroll
                for (int P = 0; P < NS; ++P) {
                    double v = 0.0;
#pragma unroll
                    for (int Q = 0; Q < NS; ++Q) v = fma(__ldg(cell + PT::NM + P * NS + Q), tp2[Q], v);
                    vc[P] = fma(-q2, __ldg(Q1 + (int64_t)i1.idx * PT::NQ + P), v);
                }
                vc[0] += prior_var;
            }
            const double t1 = (pt.x - i1.u) * mesh1.inv_delta;
            double m = mc[K];
#pragma unroll
            for (int p = K - 1; p >= 0; --p) m = fma(m, t1, mc[p]);
            double v = vc[2 * K];
#pragma unroll
            for (int P = 2 * K - 1; P >= 0; --P) v = fma(v, t1, vc[P]);
            mu = m;
            vv = v;
        };

        const uint64_t stream_policy = evict_first_policy();
        const double2* xp = X2 + r_begin * n2 + col;
        double* mp = mean + r_begin * n2 + col;
        double* vp = var + r_begin * n2 + col;
        const int64_t rows = r_end - r_begin, rows8 = rows & ~(int64_t)7;
        double2 px[8];
        if (rows8 > 0) {
#pragma unroll
            for (int u = 0; u < 8; ++u) px[u] = ldg_stream2(reinterpret_cast<const double*>(xp + u * n2), stream_policy);
        }
        for (int64_t r = 0; r < rows8; r += 8) {
            double2 cx[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) cx[u] = px[u];
            xp += 8 * n2;
            if (r + 8 < rows8) {
#pragma unroll
                for (int u = 0; u < 8; ++u) px[u] = ldg_stream2(reinterpret_cast<const double*>(xp + u * n2), stream_policy);
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                double mu, vv;
                eval(cx[u], mu, vv);
                __stcs(mp + u * n2, mu);           // written once: streaming stores keep the per-cell tables in L2
                __stcs(vp + u * n2, vv);
            }
            mp += 8 * n2;
            vp += 8 * n2;
        }
        for (int64_t r = rows8; r < rows; ++r) {
            double mu, vv;
            eval(__ldg(xp), mu, vv);
            *mp = mu;
            *vp = vv;
            xp += n2; mp += n2; vp += n2;
        }
    }
}

static int sm_count2() {
    static int cached = 0;
    if (cached == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return 148;
        if (cudaDeviceGetAttribute(&cached, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) cached = 148;
    }
    return cached;
}

// ------------------------------------------------------------------------------------------------------------------
// accumulate for inputs in no particular order: bucket partition on dimension 1 (partition.cuh), then per-unit
// shared-memory sort by cell.  (The thread-private kernel above degenerates to (2k+1)^2 + (k+1)^2 REDs per point
// once consecutive points stop sharing a cell: 35 ms per 1e8 shuffled points.)
// ------------------------------------------------------------------------------------------------------------------
constexpr int kUnitPoints2 = 4096;     // points per unit (3072-point units at two 256-thread CTAs per SM spill and measured slower: 6.46 vs 6.16 ms)
constexpr int kUnitMargin2 = 1;       // dim-1 intervals either side of a bucket the exact interval may fall into
constexpr int kUnitKnots2 = 2048;     // dim-2 knots staged in shared memory (longer meshes are read through L1)
template <int K> struct Units2 {
    // one CTA per SM: the unit's points + the exchange areas take 140..190 KB of shared memory
    static constexpr int THREADS = K <= 4 ? 512 : 256;
    static constexpr int GL = (2 * K + 1) <= 8 ? 4 : 8;                   // lanes (and points per batch) per cell; a lane owns rows l and l + GL
    static constexpr int NV = (2 * K + 1) + (K + 1);                      // factors per dimension per point
    static constexpr int NVP = (NV + 1) & ~1;                             // ... padded to whole 16-byte pairs
    static constexpr int EX = NV * GL + 2;                                // doubles of one group's exchange area (+2: groups land on different banks)
};

template <class TX, class TY>
struct Points2D {
    const TX* X;
    const TY* y;
    const double* knots1;
    int n_knots1;
    int ipb;            // dim-1 knot intervals per bucket
    double x0, inv_delta;
    __device__ __forceinline__ void init() {
        x0 = __ldg(knots1);
        inv_delta = 1.0 / (__ldg(knots1 + 1) - x0);
    }
    __device__ __forceinline__ int guess(double xv) const {
        const double g = floor((xv - x0) * inv_delta);
        const int hi = n_knots1 - 2;
        return g < 0.0 ? 0 : (g > (double)hi ? hi : (int)g);
    }
    __device__ __forceinline__ int bucket(int64_t i) const { return guess(ldg_d(X + 2 * i)) / ipb; }
    __device__ __forceinline__ void load(int64_t i, double (&v)[3]) const {
        const double2 p = ldg_point(X, i);
        v[0] = p.x; v[1] = p.y; v[2] = ldg_d(y + i);
    }
    __device__ __forceinline__ int bucket_of(const double (&v)[3]) const { return guess(v[0]) / ipb; }
};

// exact interval inside a window of knots staged in shared memory: s[j] = knot of interval first + j, j = 0..count
// (count intervals jlo..jhi are real).  Returns -1 when x lies outside the window.
__device__ __forceinline__ int locate_in_window(const double* s, int jlo, int jhi, bool open_lo, bool open_hi, double g_rel, double xv) {
    int j = (g_rel < (double)jlo) ? jlo : (g_rel > (double)jhi ? jhi : (int)g_rel);
    while (j > jlo && !(s[j] < xv)) --j;
    while (j < jhi && s[j + 1] < xv) ++j;
    const bool below = j == jlo && !open_lo && !(s[jlo] < xv);
    const bool above = j == jhi && !open_hi && s[jhi + 1] < xv;
    return (below || above) ? -1 : j;
}

// One unit = up to kUnitPoints2 records (x1, x2, y) of one bucket.  The CTA counting-sorts the unit by cell in shared
// memory ((t1, t2, y) are what is staged).  Then GL = 4 (8 for k >= 4) lanes take one cell, GL points at a time:
//   produce  lane i evaluates, for point i of the batch, the dim-1 factors A = (beta_0..2k(t1), gamma_0..k(t1)) once and
//            leaves them in the group's exchange area, transposed (row v, column i);
//   consume  lane l OWNS the moment rows with dim-1 index l and l + GL (beta_l(t1) beta_q(t2), q = 0..2k) and, for l <= k,
//            the projection row gamma_l(t1) gamma_q(t2) y: it reads its rows of A (GL values each) and evaluates the dim-2
//            factors of the GL points itself (exchanging those too made the kernel shared-memory-bandwidth-bound), one FMA
//            per moment.
// Nothing is reduced across lanes and a thread holds 5k + 3 sums instead of (2k+1)^2 + (k+1)^2; at the end of a
// cell's run each lane adds its rows to the moment table.  (Measured per 1e8 shuffled points, k = 3: 8 lanes per cell
// each recomputing every factor 5.0 ms; A and B exchanged 6.2 ms; A exchanged, 8 lanes 4.65 ms; this version 4.2 ms.)
template <int K>
__global__ void __launch_bounds__(Units2<K>::THREADS, 1)
accum_2d_units_kernel(PartWork w, int64_t n, const double* __restrict__ knots1, int nk1, const double* __restrict__ knots2,
                      int nk2, int ipb, double* __restrict__ cellmom, double* __restrict__ scal) {
    using Mo = Moments<K>;
    constexpr int NB = Mo::NB, NY = Mo::NY;
    constexpr int GL = Units2<K>::GL, EX = Units2<K>::EX;
    constexpr int THREADS = Units2<K>::THREADS;
    constexpr int PER = kUnitPoints2 / THREADS;
    constexpr int kWarps = THREADS / 32;
    const int nc2 = nk2 - 1;
    const int nb1 = ipb + 2 * kUnitMargin2;
    const int n_bins = nb1 * nc2;
    const int nk2s = nk2 < kUnitKnots2 ? nk2 : 0;           // dim-2 knots staged (0: read through L1)
    extern __shared__ double s_dyn[];
    double* s_t1 = s_dyn;                                   // [kUnitPoints2]
    double* s_t2 = s_t1 + kUnitPoints2;
    double* s_y = s_t2 + kUnitPoints2;
    double* s_ex = s_y + kUnitPoints2;                       // [THREADS / GL][EX] exchange areas
    double* s_k1 = s_ex + (THREADS / GL) * EX;              // [nb1 + 1]
    double* s_k2 = s_k1 + nb1 + 1;                          // [nk2s]
    int* s_off = reinterpret_cast<int*>(s_k2 + nk2s);       // [n_bins + 2]
    __shared__ UnitTable tab;
    __shared__ double s_yy[kWarps];
    __shared__ int s_wsum[kWarps];
    __shared__ int s_carry;
    const Mesh mesh1 = load_mesh2(knots1, nk1), mesh2 = load_mesh2(knots2, nk2);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int last1 = nk1 - 2, last2 = nk2 - 2;
    const double* r1 = w.rec;
    const double* r2 = w.rec + n;
    const double* ry = w.rec + 2 * n;
    tab.stage(w);
    for (int j = threadIdx.x; j < nk2s; j += THREADS) s_k2[j] = __ldg(knots2 + j);
    if (threadIdx.x == 0) { s_t2[0] = 0.0; s_y[0] = 0.0; }      // slot 0 stands in for points past the end of a run (times zero)
    __syncthreads();
    const int64_t n_slots = tab.n_slots();
    double yy = 0.0;
    for (int64_t u = blockIdx.x; u < n_slots; u += gridDim.x) {
        int bucket, count;
        int64_t first;
        if (!tab.find(u, kUnitPoints2, bucket, first, count)) continue;
        const int idx0 = bucket * ipb - kUnitMargin2;         // dim-1 interval of row 0 of the unit's bins
        const int jlo = idx0 < 0 ? -idx0 : 0;
        const int jhi = (last1 - idx0 < nb1 - 1) ? last1 - idx0 : nb1 - 1;
        double x1s[PER], x2s[PER], ys[PER];
#pragma unroll
        for (int p = 0; p < PER; ++p) {
            const int q = p * THREADS + threadIdx.x;
            if (q < count) { x1s[p] = __ldg(r1 + first + q); x2s[p] = __ldg(r2 + first + q); ys[p] = __ldg(ry + first + q); }
        }
        for (int j = threadIdx.x; j <= n_bins; j += THREADS) s_off[j] = 0;
        for (int j = threadIdx.x; j <= nb1; j += THREADS) {
            const int kn = idx0 + j;
            s_k1[j] = (kn >= 0 && kn < nk1) ? __ldg(knots1 + kn) : 0.0;
        }
        __syncthreads();
        int bin[PER];
#pragma unroll
        for (int p = 0; p < PER; ++p) {
            const int q = p * THREADS + threadIdx.x;
            bin[p] = -1;
            if (q < count) {
                yy = fma(ys[p], ys[p], yy);
                const double g1 = floor((x1s[p] - mesh1.x0) * mesh1.inv_delta) - (double)idx0;
                const int j1 = locate_in_window(s_k1, jlo, jhi, idx0 + jlo == 0, idx0 + jhi == last1, g1, x1s[p]);
                int c2;
                if (nk2s) {
                    const double g2 = floor((x2s[p] - mesh2.x0) * mesh2.inv_delta);
                    c2 = locate_in_window(s_k2, 0, last2, true, true, g2, x2s[p]);
                } else {
                    c2 = locate_interval(mesh2, x2s[p], LdgLoader2());
                }
                if (j1 < 0) {           // outside the unit's rows (mesh far from uniform): straight to the table
                    scatter_point_2d<K>(mesh1, mesh2, x1s[p], x2s[p], ys[p], cellmom);
                } else {
                    bin[p] = j1 * nc2 + c2;
                    atomicAdd(&s_off[bin[p] + 1], 1);
                    x1s[p] = (x1s[p] - s_k1[j1]) * mesh1.inv_delta;                        // t1
                    x2s[p] = (x2s[p] - (nk2s ? s_k2[c2] : __ldg(knots2 + c2))) * mesh2.inv_delta;   // t2
                }
            }
        }
        __syncthreads();
        // inclusive scan of s_off[1..n_bins] in place (s_off[j] becomes the first slot of bin j)
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
#pragma unroll
        for (int p = 0; p < PER; ++p) {
            if (bin[p] >= 0) {
                const int slot = atomicAdd(&s_off[bin[p]], 1);       // advances s_off[j] to the end of bin j
                s_t1[slot] = x1s[p];
                s_t2[slot] = x2s[p];
                s_y[slot] = ys[p];
            }
        }
        __syncthreads();
        // bin j is now [j ? s_off[j - 1] : 0, s_off[j]); rows outside [jlo, jhi] are empty
        const int l = lane & (GL - 1);
        double* sA = s_ex + (size_t)(threadIdx.x / GL) * EX;          // [NV][GL]
        const bool has1 = l + GL < NB, hasy = l < NY;                 // second Gram row / projection row of this lane
        const int row0 = l < NB ? l : NB - 1, row1 = has1 ? l + GL : NB - 1, row_y = NB + (hasy ? l : NY - 1);
        const int bin_lo = jlo * nc2, bin_hi = (jhi + 1) * nc2;
        for (int jb = bin_lo + warp * (32 / GL); jb < bin_hi; jb += kWarps * (32 / GL)) {
            const int j = jb + lane / GL;
            int begin = 0, end = 0;
            if (j < bin_hi) { begin = j ? s_off[j - 1] : 0; end = s_off[j]; }
            const int n_max = __reduce_max_sync(0xffffffffu, end - begin);
            if (n_max == 0) continue;
            double g0[NB], g1[NB], gy[NY];
#pragma unroll
            for (int q = 0; q < NB; ++q) { g0[q] = 0.0; g1[q] = 0.0; }
#pragma unroll
            for (int q = 0; q < NY; ++q) gy[q] = 0.0;
            for (int base = 0; base < n_max; base += GL) {
                {   // produce: the dim-1 factors of point `l` of the batch, transposed (row v, column l); zeros past the run
                    const int pt = begin + base + l;
                    const bool have = pt < end;
                    const double t1 = have ? s_t1[pt] : 0.0;
                    const double live = have ? 1.0 : 0.0;
                    double tp[2 * K + 1], up[2 * K + 1];
                    powers<2 * K>(t1, tp, up);
#pragma unroll
                    for (int v = 0; v < NB; ++v) sA[v * GL + l] = live * tp[v] * up[2 * K - v];
#pragma unroll
                    for (int v = 0; v < NY; ++v) sA[(NB + v) * GL + l] = live * tp[v] * up[K - v];
                }
                __syncwarp();
                {   // consume
                    double a0[GL], a1[GL], ay[GL];
#pragma unroll
                    for (int i = 0; i < GL; i += 2) {
                        const double2 v0 = *reinterpret_cast<const double2*>(sA + row0 * GL + i);
                        const double2 v1 = *reinterpret_cast<const double2*>(sA + row1 * GL + i);
                        const double2 vy = *reinterpret_cast<const double2*>(sA + row_y * GL + i);
                        a0[i] = v0.x; a0[i + 1] = v0.y;
                        a1[i] = has1 ? v1.x : 0.0; a1[i + 1] = has1 ? v1.y : 0.0;
                        ay[i] = vy.x; ay[i + 1] = vy.y;
                    }
                    const int left = end - begin - base;              // points of this batch that exist (may be <= 0)
#pragma unroll
                    for (int i = 0; i < GL; ++i) {
                        // past the run: slot 0, whose column of A is zero.  It must be a slot that HOLDS A FINITE NUMBER (slot 0 does:
                        // zeroed at kernel start, a real point afterwards) — a slot past the unit's count holds whatever the
                        // previous kernel left in shared memory, and 0 * NaN poisoned the cell (r02: seen once the suite's other
                        // kernels started leaving NaN bit patterns there)
                        const int pt = i < left ? begin + base + i : 0;
                        const double t2 = s_t2[pt], yv = s_y[pt];
                        double tp[2 * K + 1], up[2 * K + 1];
                        powers<2 * K>(t2, tp, up);
                        const double ayv = ay[i] * yv;
#pragma unroll
                        for (int q = 0; q < NB; ++q) {
                            const double bq = tp[q] * up[2 * K - q];
                            g0[q] = fma(a0[i], bq, g0[q]);
                            g1[q] = fma(a1[i], bq, g1[q]);
                        }
#pragma unroll
                        for (int q = 0; q < NY; ++q) gy[q] = fma(ayv, tp[q] * up[K - q], gy[q]);
                    }
                }
                __syncwarp();
            }
#ifdef ASVGP_ABLATE_RED
            double keep = 0.0;
#pragma unroll
            for (int q = 0; q < NB; ++q) keep += g0[q] + g1[q];
#pragma unroll
            for (int q = 0; q < NY; ++q) keep += gy[q];
            if (keep == 1.2345e300) {
#else
            if (end > begin) {
#endif
                const int j1 = j / nc2, c2 = j - j1 * nc2;
                double* dst = cellmom + ((int64_t)(idx0 + j1) * nc2 + c2) * Mo::kAll;
                if (l < NB) {
#pragma unroll
                    for (int q = 0; q < NB; ++q) atomicAdd(dst + l * NB + q, g0[q]);
                }
                if (has1) {
#pragma unroll
                    for (int q = 0; q < NB; ++q) atomicAdd(dst + (l + GL) * NB + q, g1[q]);
                }
                if (hasy) {
#pragma unroll
                    for (int q = 0; q < NY; ++q) atomicAdd(dst + Mo::kGram + l * NY + q, gy[q]);
                }
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) yy += __shfl_xor_sync(0xffffffffu, yy, o);
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

template <int K>
static size_t accum_2d_units_smem(int nb1, int nc2, int nk2) {
    const int nk2s = nk2 < kUnitKnots2 ? nk2 : 0;
    return (size_t)3 * kUnitPoints2 * 8 + (size_t)(Units2<K>::THREADS / Units2<K>::GL) * Units2<K>::EX * 8 +
           (size_t)(nb1 + 1 + nk2s) * 8 + (size_t)(nb1 * nc2 + 2) * 4;
}

// Fraction of sampled neighbours (point i, point i+1) that lie more than one cell apart in either dimension: ~0 for
// raster / run-ordered input, ~1 for shuffled input.
template <class TX>
__global__ void __launch_bounds__(256) order_probe_2d_kernel(const TX* __restrict__ X, int64_t n, const double* __restrict__ knots1,
                                                             int nk1, const double* __restrict__ knots2, int nk2, int samples,
                                                             double* __restrict__ out) {
    const Mesh mesh1 = load_mesh2(knots1, nk1), mesh2 = load_mesh2(knots2, nk2);
    int jumps = 0;
    for (int s = threadIdx.x; s < samples; s += blockDim.x) {
        const int64_t i = (int64_t)((double)s * (double)(n - 1) / (double)samples);
        const int a1 = locate_interval(mesh1, ldg_d(X + 2 * i), LdgLoader2()), b1 = locate_interval(mesh1, ldg_d(X + 2 * i + 2), LdgLoader2());
        const int a2 = locate_interval(mesh2, ldg_d(X + 2 * i + 1), LdgLoader2()), b2 = locate_interval(mesh2, ldg_d(X + 2 * i + 3), LdgLoader2());
        const int d1 = a1 > b1 ? a1 - b1 : b1 - a1, d2 = a2 > b2 ? a2 - b2 : b2 - a2;
        // (a raster row end — x1 moves on by at most one interval, x2 jumps back — is not a sign of disorder)
        jumps += (d1 > 1 || (d1 == 0 && d2 > 1)) ? 1 : 0;
    }
    jumps = __reduce_add_sync(0xffffffffu, jumps);
    if ((threadIdx.x & 31) == 0 && jumps) atomicAdd(out, (double)jumps / (double)samples);
}

template <int K>
static int launch_accum_2d_units(const PartWork& w, int64_t n, const double* k1, int nk1, const double* k2, int nk2, int ipb,
                                 double* cellmom, double* scal, cudaStream_t st) {
    const size_t smem = accum_2d_units_smem<K>(ipb + 2 * kUnitMargin2, nk2 - 1, nk2);
    ASVGP_REQUIRE(smem <= 227 * 1024, "accum_2d_binned: %zu bytes of shared memory needed", smem);
    ASVGP_CUDA_OK(cudaFuncSetAttribute(accum_2d_units_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    ASVGP_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, accum_2d_units_kernel<K>, Units2<K>::THREADS, smem));
    const int64_t max_units = n / kUnitPoints2 + kPartBuckets;
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(max_units, (int64_t)sm_count2() * std::max(per_sm, 1)));
    accum_2d_units_kernel<K><<<blocks, Units2<K>::THREADS, smem, st>>>(w, n, k1, nk1, k2, nk2, ipb, cellmom, scal); ASVGP_LAUNCHED();
    return kOk;
}

template <int K, int P0, int P1, bool WITH_Y, class TX, class TY>
static int launch_accum_part(const TX* X, const TY* y, int64_t n, const double* k1, int nk1, const double* k2,
                             int nk2, double* cellmom, double* scal, const int* select, cudaStream_t st) {
    const int64_t want = (n + 511) / 512;          // at least ~2 points per thread; at most one CTA per SM
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(want, sm_count2()));
    accum_2d_kernel<K, P0, P1, WITH_Y><<<blocks, 256, 0, st>>>(X, y, n, k1, nk1, k2, nk2, cellmom, scal, select, 0); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

#define PART(P0_, P1_, Y_) \
    if (rc == kOk) rc = launch_accum_part<K, P0_, P1_, Y_>(X, y, n, k1, nk1, k2, nk2, cellmom, scal, select, st);
// moment index ranges per launch: <= ~70 register-resident sums per thread
template <int K, class TX, class TY>
static int launch_accum_2d(const TX* X, const TY* y, int64_t n, const double* k1, int nk1, const double* k2,
                           int nk2, double* cellmom, double* scal, const int* select, cudaStream_t st) {
    int rc = kOk;
    if constexpr (K == 1) { PART(0, 3, true) }
    else if constexpr (K == 2) { PART(0, 5, true) }
    else if constexpr (K == 3) { PART(0, 7, true) }
    else if constexpr (K == 4) { PART(0, 5, true) PART(5, 9, false) }
    else if constexpr (K == 5) { PART(0, 3, true) PART(3, 8, false) PART(8, 11, false) }
    else { PART(0, 2, true) PART(2, 6, false) PART(6, 10, false) PART(10, 13, false) }
    return rc;
}
#undef PART

template <int K, class TX, class TY>
static int launch_cols(const TX* X, const TY* y, int64_t n, const double* k1, int nk1, const double* k2, int nk2,
                       double* cellmom, double* scal, const ProbeResult* probe, int hint_n2, cudaStream_t st) {
    constexpr size_t smem_cols = cols_smem<K, TX, TY>();
    ASVGP_CUDA_OK(cudaFuncSetAttribute(accum_2d_cols_kernel<K, TX, TY>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cols));
    const int tpw = 8;             // row segments per warp (tools/accum_sweep.py: 0.603 ms at 4, 0.581 at 8, 0.587 at 16, 0.651 at 32)
    accum_2d_cols_kernel<K, TX, TY><<<sm_count2(), kColsWarps * 32, smem_cols, st>>>(X, y, n, k1, nk1, k2, nk2, cellmom, scal, probe, hint_n2, tpw); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

template <int K, class TX, class TY>
static int launch_raster(const TX* X, const TY* y, int64_t n, const double* k1, int nk1, const double* k2, int nk2,
                         double* cellmom, double* scal, const ProbeResult* probe, int blocks, size_t smem,
                         cudaStream_t st) {
    ASVGP_CUDA_OK(cudaFuncSetAttribute(accum_2d_raster_kernel<K, true, TX, TY>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ASVGP_CUDA_OK(cudaFuncSetAttribute(accum_2d_raster_kernel<K, false, TX, TY>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    accum_2d_raster_kernel<K, true><<<blocks, kRasterWarps * 32, smem, st>>>(X, y, n, k1, nk1, k2, nk2, cellmom, scal, probe); ASVGP_LAUNCHED();
    accum_2d_raster_kernel<K, false><<<blocks, kRasterWarps * 32, smem, st>>>(X, y, n, k1, nk1, k2, nk2, cellmom, scal, probe); ASVGP_LAUNCHED();
    return launch_cols<K>(X, y, n, k1, nk1, k2, nk2, cellmom, scal, probe, 0, st);
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

extern "C" int64_t asvgp_accum_2d_moment_doubles(int n_knots1, int n_knots2, int order) {
    if (order < 1 || order > kMaxOrder || n_knots1 < 2 || n_knots2 < 2) return -1;
    const int64_t per = (int64_t)(2 * order + 1) * (2 * order + 1) + (int64_t)(order + 1) * (order + 1);
    return per * (n_knots1 - 1) * (n_knots2 - 1) + 1;          // + 1: path-selection slot of asvgp_accum_2d
}

template <class TX, class TY>
static int accum_2d_impl(const TX* X, const TY* y, int64_t n, const double* mesh1, int n_knots1, const double* mesh2,
                         int n_knots2, int order, double* cellmom, double* scal, cudaStream_t st) {
    // Path selection without a host round trip: a one-CTA probe classifies the input (raster / x1-runs / general) into
    // the trailing slot of the moment table (asvgp_accum_2d_moment_doubles reserves it); every candidate kernel is
    // launched and those that are not selected return at once.
    ProbeResult* probe = reinterpret_cast<ProbeResult*>(cellmom + asvgp_accum_2d_moment_doubles(n_knots1, n_knots2, order) - 1);
    const int* select = &probe->select;
    accum_2d_probe_kernel<<<1, 1024, 0, st>>>(X, y, n, probe); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    const int blocks2 = 2 * sm_count2();
    const size_t raster_smem = sizeof(double) * 2 * kRasterWarps * 32 * (3 * (size_t)order + 2);   // NS = (2k+1) + (k+1)
    ASVGP_DISPATCH_ORDER(order, { if (int rc = launch_raster<K>(X, y, n, mesh1, n_knots1, mesh2, n_knots2, cellmom, scal, probe, blocks2, raster_smem, st)) return rc; });
    ASVGP_CUDA_OK(cudaGetLastError());
    {
        const int64_t want = (n + 1023) / 1024;
        const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)blocks2));
        ASVGP_DISPATCH_ORDER(order, (accum_2d_run_kernel<K><<<blocks, 256, 0, st>>>(X, y, n, mesh1, n_knots1, mesh2, n_knots2, cellmom, scal, select, 1))); ASVGP_LAUNCHED();
        ASVGP_CUDA_OK(cudaGetLastError());
    }
    ASVGP_DISPATCH_ORDER(order, { if (int rc = launch_accum_2d<K>(X, y, n, mesh1, n_knots1, mesh2, n_knots2, cellmom, scal, select, st)) return rc; });
    return kOk;
}

extern "C" int asvgp_accum_2d_typed(const void* X, int x_type, const void* y, int y_type, int64_t n, const double* mesh1,
                                    int n_knots1, const double* mesh2, int n_knots2, int order, double* cellmom, double* scal,
                                    void* stream) {
    ASVGP_REQUIRE_TYPES("accum_2d", x_type, y_type);
    ASVGP_REQUIRE(n >= 0 && n_knots1 >= 2 && n_knots2 >= 2, "accum_2d: n=%lld knots=%d,%d", (long long)n, n_knots1, n_knots2);
    ASVGP_REQUIRE((reinterpret_cast<uintptr_t>(X) & 15u) == 0 && (reinterpret_cast<uintptr_t>(y) & 15u) == 0,
                  "accum_2d: X and y must be 16-byte aligned");
    if (n == 0) return kOk;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    return with_elem_types(x_type, y_type, [&](auto tx, auto ty) -> int {
        using TX = typename decltype(tx)::type;
        using TY = typename decltype(ty)::type;
        return accum_2d_impl(static_cast<const TX*>(X), static_cast<const TY*>(y), n, mesh1, n_knots1, mesh2, n_knots2, order,
                             cellmom, scal, st);
    });
}

extern "C" int asvgp_accum_2d(const double* X, const double* y, int64_t n, const double* mesh1, int n_knots1,
                              const double* mesh2, int n_knots2, int order, double* cellmom, double* scal,
                              void* stream) {
    return asvgp_accum_2d_typed(X, ASVGP_F64, y, ASVGP_F64, n, mesh1, n_knots1, mesh2, n_knots2, order, cellmom, scal, stream);
}

extern "C" int asvgp_accum_2d_raster_typed(const void* X, int x_type, const void* y, int y_type, int64_t n, int64_t row_len,
                                           const double* mesh1, int n_knots1, const double* mesh2, int n_knots2, int order,
                                           double* cellmom, double* scal, void* stream) {
    ASVGP_REQUIRE_TYPES("accum_2d_raster", x_type, y_type);
    ASVGP_REQUIRE(n >= 0 && n_knots1 >= 2 && n_knots2 >= 2, "accum_2d_raster: n=%lld knots=%d,%d", (long long)n, n_knots1, n_knots2);
    ASVGP_REQUIRE(row_len > 0 && row_len <= 0x7fffffff && n % row_len == 0, "accum_2d_raster: n=%lld is not a whole number of rows of %lld points",
                  (long long)n, (long long)row_len);
    ASVGP_REQUIRE((reinterpret_cast<uintptr_t>(X) & 15u) == 0 && (reinterpret_cast<uintptr_t>(y) & 15u) == 0,
                  "accum_2d_raster: X and y must be 16-byte aligned");
    if (n == 0) return kOk;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    return with_elem_types(x_type, y_type, [&](auto tx, auto ty) -> int {
        using TX = typename decltype(tx)::type;
        using TY = typename decltype(ty)::type;
        const TX* Xt = static_cast<const TX*>(X);
        const TY* yt = static_cast<const TY*>(y);
        ASVGP_DISPATCH_ORDER(order, { if (int rc = launch_cols<K>(Xt, yt, n, mesh1, n_knots1, mesh2, n_knots2, cellmom, scal, nullptr, (int)row_len, st)) return rc; });
        return kOk;
    });
}

extern "C" int asvgp_accum_2d_raster(const double* X, const double* y, int64_t n, int64_t row_len, const double* mesh1,
                                     int n_knots1, const double* mesh2, int n_knots2, int order, double* cellmom,
                                     double* scal, void* stream) {
    return asvgp_accum_2d_raster_typed(X, ASVGP_F64, y, ASVGP_F64, n, row_len, mesh1, n_knots1, mesh2, n_knots2, order, cellmom,
                                       scal, stream);
}

extern "C" int64_t asvgp_accum_2d_binned_work_bytes(int64_t n) { return PartWork::bytes(n < 0 ? 0 : n, 3); }

extern "C" int asvgp_order_probe_2d_typed(const void* X, int x_type, int64_t n, const double* mesh1, int n_knots1,
                                          const double* mesh2, int n_knots2, double* out, void* stream) {
    ASVGP_REQUIRE(valid_elem_type(x_type), "order_probe_2d: element type %d (0 = float64, 1 = float32)", x_type);
    ASVGP_REQUIRE(n >= 0 && n_knots1 >= 2 && n_knots2 >= 2 && out != nullptr, "order_probe_2d: n=%lld knots=%d,%d",
                  (long long)n, n_knots1, n_knots2);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ASVGP_CUDA_OK(cudaMemsetAsync(out, 0, sizeof(double), st));
    if (n < 2) return kOk;
    const int samples = (int)std::min<int64_t>(n - 1, 4096);
    if (x_type == ASVGP_F32) order_probe_2d_kernel<<<1, 256, 0, st>>>(static_cast<const float*>(X), n, mesh1, n_knots1, mesh2, n_knots2, samples, out);
    else order_probe_2d_kernel<<<1, 256, 0, st>>>(static_cast<const double*>(X), n, mesh1, n_knots1, mesh2, n_knots2, samples, out);
    ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

extern "C" int asvgp_order_probe_2d(const double* X, int64_t n, const double* mesh1, int n_knots1, const double* mesh2,
                                    int n_knots2, double* out, void* stream) {
    return asvgp_order_probe_2d_typed(X, ASVGP_F64, n, mesh1, n_knots1, mesh2, n_knots2, out, stream);
}

extern "C" int asvgp_accum_2d_binned_typed(const void* X, int x_type, const void* y, int y_type, int64_t n, const double* mesh1,
                                           int n_knots1, const double* mesh2, int n_knots2, int order, double* cellmom,
                                           double* scal, void* work, int64_t work_bytes, void* stream) {
    ASVGP_REQUIRE_TYPES("accum_2d_binned", x_type, y_type);
    ASVGP_REQUIRE(n >= 0 && n_knots1 >= 2 && n_knots2 >= 2, "accum_2d_binned: n=%lld knots=%d,%d", (long long)n, n_knots1, n_knots2);
    ASVGP_REQUIRE(order >= 1 && order <= kMaxOrder, "accum_2d_binned: spline order %d not in 1..6", order);
    ASVGP_REQUIRE((reinterpret_cast<uintptr_t>(X) & 15u) == 0, "accum_2d_binned: X must be 16-byte aligned");
    const int nc1 = n_knots1 - 1, nc2 = n_knots2 - 1;
    const int ipb = (nc1 + kPartBuckets - 1) / kPartBuckets;
    size_t smem_units = 0;
    ASVGP_DISPATCH_ORDER(order, (smem_units = accum_2d_units_smem<K>(ipb + 2 * kUnitMargin2, nc2, n_knots2)));
    // too many cells per bucket for the shared-memory sort: the streaming kernels handle any order
    if ((int64_t)(ipb + 2 * kUnitMargin2) * nc2 > kUnitMaxBins || smem_units > 227 * 1024)
        return asvgp_accum_2d_typed(X, x_type, y, y_type, n, mesh1, n_knots1, mesh2, n_knots2, order, cellmom, scal, stream);
    ASVGP_REQUIRE(work != nullptr && work_bytes >= PartWork::bytes(n, 3), "accum_2d_binned: work_bytes=%lld < %lld",
                  (long long)work_bytes, (long long)PartWork::bytes(n, 3));
    if (n == 0) return kOk;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const PartWork w = PartWork::carve(work);
    ASVGP_CUDA_OK(cudaMemsetAsync(w.count, 0, kPartBuckets * sizeof(u64), st));
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((n + kPartTile - 1) / kPartTile, (int64_t)sm_count2() * 2));
    // the partition reads the points in their own types and writes float64 records: the units kernel is type-free
    const int prc = with_elem_types(x_type, y_type, [&](auto tx, auto ty) -> int {
        using TX = typename decltype(tx)::type;
        using TY = typename decltype(ty)::type;
        Points2D<TX, TY> src;
        src.X = static_cast<const TX*>(X); src.y = static_cast<const TY*>(y); src.knots1 = mesh1; src.n_knots1 = n_knots1; src.ipb = ipb;
        ASVGP_CUDA_OK((launch_partition<Points2D<TX, TY>, 3>(src, n, w, kUnitPoints2, blocks, st)));
        return kOk;
    });
    if (prc != kOk) return prc;
    ASVGP_DISPATCH_ORDER(order, { if (int rc = launch_accum_2d_units<K>(w, n, mesh1, n_knots1, mesh2, n_knots2, ipb, cellmom, scal, st)) return rc; });
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

extern "C" int asvgp_accum_2d_binned(const double* X, const double* y, int64_t n, const double* mesh1, int n_knots1,
                                     const double* mesh2, int n_knots2, int order, double* cellmom, double* scal,
                                     void* work, int64_t work_bytes, void* stream) {
    return asvgp_accum_2d_binned_typed(X, ASVGP_F64, y, ASVGP_F64, n, mesh1, n_knots1, mesh2, n_knots2, order, cellmom, scal, work,
                                       work_bytes, stream);
}

extern "C" int asvgp_expand_moments_2d(const double* cellmom, const double* Cprod, const double* Dy, int n_knots1,
                                       int n_knots2, int order, double* Gs, double* b, void* stream) {
    ASVGP_REQUIRE(n_knots1 >= 2 && n_knots2 >= 2, "expand_moments_2d: knots=%d,%d", n_knots1, n_knots2);
    const int nc1 = n_knots1 - 1, nc2 = n_knots2 - 1;
    const int m2 = n_knots2 + order - 1;
    const int64_t M = (int64_t)(n_knots1 + order - 1) * m2;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int blocks = std::min(nc1 * nc2, sm_count2() * 8);
    ASVGP_DISPATCH_ORDER(order, (expand_moments_2d_kernel<K><<<blocks, 256, 0, st>>>(cellmom, Cprod, Dy, nc1, nc2, m2, M, Gs, b))); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

extern "C" int64_t asvgp_predict_2d_work_doubles(int n_knots1, int n_knots2, int order) {
    if (order < 1 || order > kMaxOrder || n_knots1 < 2 || n_knots2 < 2) return -1;
    const int64_t nc1 = n_knots1 - 1, nc2 = n_knots2 - 1;
    const int64_t cell = (int64_t)(order + 1) * (order + 1) + (int64_t)(2 * order + 1) * (2 * order + 1);
    return nc1 * nc2 * cell + (nc1 + nc2) * (2 * order + 1) + 1;        // + 1: slot of the input classification probe
}

template <int K>
static int launch_predict_2d_prepare(int nk1, int nk2, const double* alpha, const double* SigP, const double* S1, const double* S2,
                                     double* work, cudaStream_t st) {
    const int nc1 = nk1 - 1, nc2 = nk2 - 1, m1 = nk1 + K - 1, m2 = nk2 + K - 1;
    constexpr int W = (K + 1) * (K + 1);
    const size_t smem = sizeof(double) * (size_t)(W * W + W + W * (2 * K + 1));      // window, alpha, stage-1 result
    ASVGP_CUDA_OK(cudaFuncSetAttribute(predict_2d_table_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    predict_2d_table_kernel<K><<<nc1 * nc2 + 2, 256, smem, st>>>(nc1, nc2, m1, m2, alpha, SigP, S1, S2, work); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

template <int K>
static int launch_predict_2d_apply(const double* Xnew, int64_t n, int hint_n2, const double* mesh1, int nk1, const double* mesh2,
                                   int nk2, double prior_var, double* mean, double* var, double* work, cudaStream_t st) {
    ProbeResult* probe = reinterpret_cast<ProbeResult*>(work + asvgp_predict_2d_work_doubles(nk1, nk2, K) - 1);
    const int cols_mult = 6;       // CTAs per SM's worth of tasks (tools/predict_2d_sweep.py: 0.69 ms at 2, 0.64 ms at 6, 0.66 ms at 8)
    if (hint_n2 > 0) {      // the caller states the test set is a flattened raster: column sweep only (it re-checks every point)
        predict_2d_cols_kernel<K><<<cols_mult * sm_count2(), 256, 0, st>>>(Xnew, n, mesh1, nk1, mesh2, nk2, work, prior_var, mean, var, probe, hint_n2); ASVGP_LAUNCHED();
        ASVGP_CUDA_OK(cudaGetLastError());
        return kOk;
    }
    // classification probe (as in asvgp_accum_2d): separable raster test sets take the coalesced column sweep, anything else
    // the thread-contiguous kernel; the one that is not selected returns at once
    accum_2d_probe_kernel<<<1, 1024, 0, st>>>(Xnew, Xnew, n, probe); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    predict_2d_cols_kernel<K><<<cols_mult * sm_count2(), 256, 0, st>>>(Xnew, n, mesh1, nk1, mesh2, nk2, work, prior_var, mean, var, probe, 0); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    const bool vec = ((reinterpret_cast<uintptr_t>(Xnew) | reinterpret_cast<uintptr_t>(mean) | reinterpret_cast<uintptr_t>(var)) & 31u) == 0;
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((n + 1023) / 1024, 2 * (int64_t)sm_count2()));
    if (vec) predict_2d_kernel<K, true><<<blocks, 256, 0, st>>>(Xnew, n, mesh1, nk1, mesh2, nk2, work, prior_var, mean, var, probe);
    else predict_2d_kernel<K, false><<<blocks, 256, 0, st>>>(Xnew, n, mesh1, nk1, mesh2, nk2, work, prior_var, mean, var, probe);
    ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

extern "C" int asvgp_predict_2d_prepare(int n_knots1, int n_knots2, int order, const double* alpha, const double* SigP,
                                        const double* S1, const double* S2, double* work, void* stream) {
    ASVGP_REQUIRE(n_knots1 >= 2 && n_knots2 >= 2, "predict_2d_prepare: knots=%d,%d", n_knots1, n_knots2);
    ASVGP_REQUIRE(work != nullptr, "predict_2d_prepare: work buffer (asvgp_predict_2d_work_doubles) is required");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ASVGP_DISPATCH_ORDER(order, { if (int rc = launch_predict_2d_prepare<K>(n_knots1, n_knots2, alpha, SigP, S1, S2, work, st)) return rc; });
    return kOk;
}

extern "C" int asvgp_predict_2d_apply(const double* Xnew, int64_t n, int64_t row_len, const double* mesh1, int n_knots1,
                                      const double* mesh2, int n_knots2, int order, double prior_var, double* mean,
                                      double* var, double* work, void* stream) {
    ASVGP_REQUIRE(n >= 0 && n_knots1 >= 2 && n_knots2 >= 2, "predict_2d_apply: n=%lld", (long long)n);
    ASVGP_REQUIRE((reinterpret_cast<uintptr_t>(Xnew) & 15u) == 0, "predict_2d_apply: Xnew must be 16-byte aligned");
    ASVGP_REQUIRE(work != nullptr, "predict_2d_apply: work buffer prepared by asvgp_predict_2d_prepare is required");
    ASVGP_REQUIRE(row_len >= 0 && row_len <= 0x7fffffff && (row_len == 0 || n % row_len == 0),
                  "predict_2d_apply: n=%lld is not a whole number of rows of %lld points", (long long)n, (long long)row_len);
    if (n == 0) return kOk;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ASVGP_DISPATCH_ORDER(order, { if (int rc = launch_predict_2d_apply<K>(Xnew, n, (int)row_len, mesh1, n_knots1, mesh2, n_knots2, prior_var, mean, var, work, st)) return rc; });
    return kOk;
}

extern "C" int asvgp_predict_2d(const double* Xnew, int64_t n, const double* mesh1, int n_knots1, const double* mesh2,
                                int n_knots2, int order, const double* alpha, const double* SigP, const double* S1,
                                const double* S2, double prior_var, double* mean, double* var, double* work,
                                void* stream) {
    ASVGP_REQUIRE(n >= 0 && n_knots1 >= 2 && n_knots2 >= 2, "predict_2d: n=%lld", (long long)n);
    ASVGP_REQUIRE((reinterpret_cast<uintptr_t>(Xnew) & 15u) == 0, "predict_2d: Xnew must be 16-byte aligned");
    ASVGP_REQUIRE(work != nullptr, "predict_2d: work buffer (asvgp_predict_2d_work_doubles) is required");
    if (n == 0) return kOk;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (int rc = asvgp_predict_2d_prepare(n_knots1, n_knots2, order, alpha, SigP, S1, S2, work, stream)) return rc;
    ASVGP_DISPATCH_ORDER(order, { if (int rc = launch_predict_2d_apply<K>(Xnew, n, 0, mesh1, n_knots1, mesh2, n_knots2, prior_var, mean, var, work, st)) return rc; });
    return kOk;
}
