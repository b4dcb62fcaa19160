// Shared device/host helpers of libasvgp_sm100a: error reporting, knot-interval location, B-spline pieces.
//
// Everything numeric here is `ASVGP_HD` (host + device) so that tests/host_harness.cpp can compile the very same
// templates with g++ and check them against numpy on a machine without a GPU.  That harness is test
// infrastructure; the product entry points (the extern "C" functions) only ever launch the CUDA kernels.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cmath>

#if defined(__CUDACC__)
#define ASVGP_HD __host__ __device__ __forceinline__
#else
#define ASVGP_HD inline
#endif

namespace asvgp {

constexpr int kMaxOrder = 6;

// ---- status codes returned by every C-ABI entry point (0 = ok, <0 = bad argument / CUDA error) ----------------
enum Status : int {
    kOk = 0,
    kBadArgument = -1,
    kCudaError = -2,
    kUnsupported = -3,
};

void set_last_error(const char* fmt, ...);
// every kernel launch of the library is counted (asvgp_launch_count(): what bench.py reports as `gpu_launches`)
void count_launch();
#define ASVGP_LAUNCHED() ::asvgp::count_launch()

#if defined(__CUDACC__)
#define ASVGP_CUDA_OK(expr)                                                                         \
    do {                                                                                            \
        cudaError_t err__ = (expr);                                                                 \
        if (err__ != cudaSuccess) {                                                                 \
            ::asvgp::set_last_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(err__),      \
                                    __FILE__, __LINE__);                                            \
            return ::asvgp::kCudaError;                                                             \
        }                                                                                           \
    } while (0)
#endif

#define ASVGP_REQUIRE(cond, ...)                      \
    do {                                              \
        if (!(cond)) {                                \
            ::asvgp::set_last_error(__VA_ARGS__);     \
            return ::asvgp::kBadArgument;             \
        }                                             \
    } while (0)

// ---- knot mesh ------------------------------------------------------------------------------------------------
// The kernels take the mesh *array* (not just a, delta): the reference gathers the left knot u from the mesh and
// uses delta = mesh[1]-mesh[0] for every interval (basis.py:18,58-59), and a TF-built float32 mesh has slightly
// uneven gaps (SURVEY quirks Q1-Q3).
struct Mesh {
    const double* knots;   // [n_knots], ascending
    int n_knots;           // m - k + 1
    double x0;             // knots[0]
    double inv_delta;      // 1 / (knots[1] - knots[0])
};

#if defined(__CUDACC__)
// Streaming loads of the points: read once, so they are marked evict-first in L2 — they must not push out what is reused (the
// band or moment table being accumulated into, predictor tables, the tables of a Kuu chain running beside the kernel).
__device__ __forceinline__ uint64_t evict_first_policy() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ double2 ldg_stream2(const double* p, uint64_t pol) {
    double2 v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.f64 {%0, %1}, [%2], %3;" : "=d"(v.x), "=d"(v.y) : "l"(p), "l"(pol));
    return v;
}

__device__ __forceinline__ float4 ldg_stream4f(const float* p, uint64_t pol) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol));
    return v;
}

__device__ __forceinline__ void cp_async_16_stream(unsigned dst_smem, const void* src, uint64_t pol) {
    asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2;" ::"r"(dst_smem), "l"(src), "l"(pol) : "memory");
}
__device__ __forceinline__ void cp_async_8_stream(unsigned dst_smem, const void* src, uint64_t pol) {
    asm volatile("cp.async.ca.shared.global.L2::cache_hint [%0], [%1], 8, %2;" ::"r"(dst_smem), "l"(src), "l"(pol) : "memory");
}
__device__ __forceinline__ void cp_async_4_stream(unsigned dst_smem, const void* src, uint64_t pol) {
    asm volatile("cp.async.ca.shared.global.L2::cache_hint [%0], [%1], 4, %2;" ::"r"(dst_smem), "l"(src), "l"(pol) : "memory");
}
#endif

// ---- element types of the training points (ASVGP_F64 / ASVGP_F32 of the C ABI) ----------------------------------------
// The point-reading kernels are templated on the element types of x / X and y and convert every loaded value to double in
// registers (exact for float), so all arithmetic after the load is the float64 code.
template <class T> struct TypeTag { using type = T; };
ASVGP_HD bool valid_elem_type(int t) { return t == 0 || t == 1; }
// the element-type check of a typed entry point taking two arrays (before any CUDA call)
#define ASVGP_REQUIRE_TYPES(what, xt, yt) \
    ASVGP_REQUIRE(::asvgp::valid_elem_type(xt) && ::asvgp::valid_elem_type(yt), \
                  what ": element types %d, %d (0 = float64, 1 = float32)", xt, yt)
// f(TypeTag<TX>(), TypeTag<TY>()) for the two type codes (checked with valid_elem_type beforehand)
template <class F>
int with_elem_types(int x_type, int y_type, F&& f) {
    if (x_type == 1) return y_type == 1 ? f(TypeTag<float>(), TypeTag<float>()) : f(TypeTag<float>(), TypeTag<double>());
    return y_type == 1 ? f(TypeTag<double>(), TypeTag<float>()) : f(TypeTag<double>(), TypeTag<double>());
}

template <class LoadFn>
ASVGP_HD int locate_interval(const Mesh& mesh, double x, LoadFn load) {
    // Reference semantics (basis.py:58): idx = max(searchsorted_left(mesh, x) - 1, 0), i.e. the largest idx with
    // mesh[idx] < x (a point exactly on a knot belongs to the interval on its LEFT, quirk Q2); clamped to the
    // last interval for x >= b (the reference would index one row past the matrix there, quirk Q4).
    int hi = mesh.n_knots - 2;
    double g = floor((x - mesh.x0) * mesh.inv_delta);
    int idx = g < 0.0 ? 0 : (g > (double)hi ? hi : (int)g);
    while (idx > 0 && !(load(mesh.knots + idx) < x)) --idx;
    while (idx < hi && load(mesh.knots + idx + 1) < x) ++idx;
    return idx;
}

// ---- B-spline pieces --------------------------------------------------------------------------------------------
// w[r], r = 0..K : value at t = (x-u)/delta of basis row idx + r on interval idx (reference b_{K+1-r},
// basis.py:72,133-136,188-192,274-280,...): piece_r(t) = N_K(t + K - r), N_K the cardinal B-spline.
//
// The piece polynomials are generated at COMPILE time: K! * N_K(s + t) has integer coefficients, built by the
// Cox-de Boor recursion  d! N_d(s+t) = (t+s) (d-1)! N_{d-1}(s+t) + (d+1-s-t) (d-1)! N_{d-1}(s-1+t)  in integer
// arithmetic, so every coefficient c/K! is a correctly rounded double and each piece costs K FMAs (Horner) —
// K(K+1) fp64 instructions per point instead of ~5x that for the recursion evaluated at run time (the accumulate
// kernel was fp64-pipe bound with the latter: profiles/r01_accum_1d_v1.md).
template <int K>
struct PieceTable {
    long long c[K + 1][K + 1];   // c[r][p]: coefficient of t^p in K! * piece_r(t)
    long long fact;              // K!
};

template <int K>
constexpr PieceTable<K> make_piece_table() {
    long long prev[K + 1][K + 2] = {};
    long long cur[K + 1][K + 2] = {};
    prev[0][0] = 1;
    long long fact = 1;
    for (int d = 1; d <= K; ++d) {
        fact *= d;
        for (int s = 0; s <= d; ++s)
            for (int p = 0; p <= K + 1; ++p) cur[s][p] = 0;
        for (int s = 0; s <= d; ++s) {
            if (s <= d - 1)
                for (int p = 0; p <= d - 1; ++p) { cur[s][p] += s * prev[s][p]; cur[s][p + 1] += prev[s][p]; }
            if (s >= 1)
                for (int p = 0; p <= d - 1; ++p) { cur[s][p] += (d + 1 - s) * prev[s - 1][p]; cur[s][p + 1] -= prev[s - 1][p]; }
        }
        for (int s = 0; s <= d; ++s)
            for (int p = 0; p <= K + 1; ++p) prev[s][p] = cur[s][p];
    }
    PieceTable<K> t{};
    t.fact = fact;
    for (int r = 0; r <= K; ++r)
        for (int p = 0; p <= K; ++p) t.c[r][p] = prev[K - r][p];
    return t;
}

template <int K>
ASVGP_HD void bspline_pieces(double t, double (&w)[K + 1]) {
    constexpr PieceTable<K> tab = make_piece_table<K>();
#pragma unroll
    for (int r = 0; r <= K; ++r) {
        double acc = (double)tab.c[r][K] / (double)tab.fact;
#pragma unroll
        for (int p = K - 1; p >= 0; --p) acc = fma(acc, t, (double)tab.c[r][p] / (double)tab.fact);
        w[r] = acc;
    }
}

// dx-th derivative pieces by Horner on the exact piece coefficients (host-provided, (K+1)x(K+1) row-major,
// ascending powers of t), scaled by delta^-dx.  Only used by the API-parity entry point asvgp_basis_eval_1d.
template <int K>
ASVGP_HD void bspline_pieces_coef(double t, const double* coef, double scale, double (&w)[K + 1]) {
#pragma unroll
    for (int r = 0; r <= K; ++r) {
        double acc = coef[r * (K + 1) + K];
#pragma unroll
        for (int p = K - 1; p >= 0; --p) acc = acc * t + coef[r * (K + 1) + p];
        w[r] = acc * scale;
    }
}

ASVGP_HD constexpr int tri_index(int r, int s) { return r * (r + 1) / 2 + s; }   // r >= s
template <int K> struct Counts {
    static constexpr int kPairs = (K + 1) * (K + 2) / 2;   // unique entries of w w^T
    static constexpr int kAcc = kPairs + (K + 1);          // + projections w*y
};

// ---- centred monomial moments ----------------------------------------------------------------------------------------
// Every product piece_r(t) piece_s(t) is a polynomial of degree 2K in tau = t - 1/2 and every piece_r(t) one of degree K,
// so the per-interval sums of w w^T and w y follow from the 2K+1 moments  sum tau^j  and the K+1 moments  sum y tau^j:
// 5K+2 fp64 instructions per point instead of the K(K+1) + (K+1)(K+4)/2 of evaluating the pieces and their products
// (17 vs 26 for K = 3), and fewer registers.  Centring keeps the conversion benign: |tau| <= 1/2, so the terms of
// sum_j e_j M_j decay like 2^-j and cancel by at most an order of magnitude (parity at 1e-10 has four digits to spare).
// The conversion coefficients are exact integers over (K! 2^K)^2 resp. K! 2^K, built at compile time:
//     K! 2^K piece_r(tau + 1/2) = sum_q d[r][q] tau^q,   d[r][q] = sum_{p>=q} c[r][p] C(p,q) 2^(K-p+q).
template <int K>
struct MomentCoef {
    double cg[Counts<K>::kPairs][2 * K + 1];   // sum_n w_r w_s = sum_j cg[tri(r,s)][j] * M_j,  M_j = sum_n tau^j
    double cb[K + 1][K + 1];                   // sum_n w_r y   = sum_j cb[r][j] * Y_j,         Y_j = sum_n y tau^j
    int rr[Counts<K>::kPairs], ss[Counts<K>::kPairs];
};

template <int K>
constexpr MomentCoef<K> make_moment_coef() {
    const PieceTable<K> tab = make_piece_table<K>();
    long long binom[K + 1][K + 1] = {};
    for (int n = 0; n <= K; ++n) {
        binom[n][0] = 1;
        for (int k = 1; k <= n; ++k) binom[n][k] = binom[n - 1][k - 1] + (k <= n - 1 ? binom[n - 1][k] : 0);
    }
    long long d[K + 1][K + 1] = {};
    for (int r = 0; r <= K; ++r)
        for (int q = 0; q <= K; ++q) {
            long long acc = 0;
            for (int p = q; p <= K; ++p) acc += tab.c[r][p] * binom[p][q] * (1LL << (K - p + q));
            d[r][q] = acc;
        }
    const double den = (double)tab.fact * (double)(1LL << K);
    MomentCoef<K> m{};
    for (int r = 0; r <= K; ++r) {
        for (int q = 0; q <= K; ++q) m.cb[r][q] = (double)d[r][q] / den;
        for (int s = 0; s <= r; ++s) {
            const int idx = tri_index(r, s);
            m.rr[idx] = r;
            m.ss[idx] = s;
            for (int j = 0; j <= 2 * K; ++j) {
                long long acc = 0;
                for (int q = 0; q <= K; ++q) {
                    const int q2 = j - q;
                    if (q2 >= 0 && q2 <= K) acc += d[r][q] * d[s][q2];
                }
                m.cg[idx][j] = (double)acc / (den * den);
            }
        }
    }
    return m;
}
#if defined(__CUDACC__)
template <int K> __device__ const MomentCoef<K> g_moment_coef = make_moment_coef<K>();
#endif

}  // namespace asvgp
