// Nested-dissection multifrontal factorisation and selected inverse of the 2-D (Kronecker) model's
//     P = K1 (x) K2 + KufKfu / sigma2        (reference gpr.py:292; m1 m2 x m1 m2, a DENSE tf.linalg.cholesky there)
//
//   asvgp_kron_factor  <- utils.bands_to_kron_cholesky's Kronecker product, `Kuu + KufKfu / sigma2`,
//                         tf.linalg.cholesky(P), its log-det, triangular_solve(L_P, Kuf_y)            (gpr.py:287-295)
//   asvgp_kron_selinv  <- what TF reverse mode / cholesky_solve extract from P^-1 (gpr.py:307, 319-326): the entries of
//                         P^-1 on the stencil pattern and P^-1 Kuf_y
//
// Why not the band.  In the natural order P is a band of scalar width k (m2 + 1) (gpr.py:262) and its Cholesky is ONE
// dependency chain over all m1 m2 columns: 625 block columns of 64 at 200 x 200, 34 us each, with 98 % of the GPU idle
// (tiledag_2d.cu, kept as asvgp_kronband_*).  The coupling graph, however, is a 2-D grid with a (2k+1) x (2k+1) stencil:
// a strip of k grid lines separates it.  Recursive bisection by such strips (nested dissection) turns the factorisation
// into a tree of dense FRONTS — separator unknowns + the ancestors' separator unknowns they touch — in which all fronts
// of one tree level are independent and the dependency chain is the sum of the separator sizes along ONE root-to-leaf
// path: 601 + 297 + 297 + 144 + 144 + 69 + 69 + 30 + 100 = 1751 columns (33 block columns) instead of 40 000 (625), for
// 2.6x fewer flops as well.  tools/nd_prototype.py is the same algorithm in numpy (checked against LAPACK's band
// routines in tests/test_nd_plan.py).
//
// Data.  Front f has ns separator unknowns (eliminated here) and nb boundary unknowns (ancestors), each padded to a
// multiple of 64 (separator padding = unit diagonal, boundary padding = zero rows); its lower triangle is stored as
// 64 x 64 column-major tiles packed by block column, so one TMA bulk copy fetches an operand (as in tiledag_2d.cu).
// The right-hand side Kuf_y rides along as ONE EXTRA BOUNDARY UNKNOWN of every front ("rhs node", never eliminated):
// row rhs of L is y^T = (L^-1 b)^T, the root's update entry (rhs, rhs) is -||y||^2, and seeding the selected inverse
// with Sigma'(rhs, rhs) = tau gives Sigma'(s, rhs) = -tau x, x = P^-1 b, and Sigma' = P^-1 + tau x x^T on the grid
// unknowns (inverse of [[P, b], [b^T, ||y||^2 + 1/tau]]); tau = 2^-20 / (1 + ||y||^2) keeps the correction tau x x^T a
// 1e-6 fraction of sqrt(P^-1_ii P^-1_jj) (Cauchy-Schwarz), so subtracting it costs no digits.  No separate triangular
// solves, no separate chains.
//
// Several right-hand sides (multi-output targets, the *_multi entry points).  B = [b_1 ... b_D] rides along as D rhs nodes
// with ids M ... M+D-1, the last D boundary unknowns of every front; the root's boundary is exactly these D ids (one tile).
// The factorised matrix is A' = [[P, B], [B^T, 0]]: eliminating the grid unknowns leaves the root update block -B^T P^-1 B,
// whose diagonal is -Q_d, Q_d = b_d^T P^-1 b_d.  Seeding the selected inverse with Sigma'(rhs, rhs) = tau I_D gives
// Sigma'(s, rhs_d) = -tau x_d, x_d = P^-1 b_d, and Sigma' = P^-1 + tau sum_d x_d x_d^T on the grid, so the stencil of P^-1
// and the dense A^-1 are Sigma' - tau sum_d x_d x_d^T.  tau = 2^-20 / (1 + sum_d Q_d) (today's tau for D = 1) keeps the
// correction below 2^-20 sqrt(P^-1_ii P^-1_jj): |x_d,i| <= sqrt(P^-1_ii Q_d) by Cauchy-Schwarz.  One factorisation and one
// selected inverse serve every column; with D = 1 the plan and every operation are those of the single-rhs functions.
//
// Kernels, per tree level (bottom-up for the factorisation, top-down for the selected inverse):
//   nd_assemble_kernel   (once) entries of P and the right-hand-side row into every front
//   nd_factor_kernel     persistent tile DAG over all tiles of all fronts of the level: left-looking updates on the fp64
//                        tensor cores, diagonal tiles factorised + inverted in registers; trailing tiles = this front's update
//                        matrix, added straight into the parent's front (extend-add as fp64 REDs, off the chain of diagonal tiles)
//   nd_ypass_kernel      (once) L(R,C) -> Y(R,C)^T = (L(R,C) L(C,C)^-1)^T, Sigma(C,C) seeded with L(C,C)^-T L(C,C)^-1
//   nd_gather_kernel     Sigma on the boundary of a front from its parent's Sigma
//   nd_selinv_kernel     persistent tile DAG: blocked Takahashi recursion inside every front of the level
//   nd_scalars_kernel / nd_x_kernel / nd_stencil_kernel   log|P|, ||y_d||^2, x_d, stencil entries of P^-1
#include <cstdlib>
#include <map>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "tile_ops.cuh"
#include "../../include/asvgp_b200.h"

namespace asvgp {

// ---------------------------------------------------------------------------------------------------------------------
// symbolic plan (host, built once per (m1, m2, order, device) and cached with its device copies)
// ---------------------------------------------------------------------------------------------------------------------
struct FrontDesc {                 // device-visible
    long long tile_base;           // first tile of this front in the tile pools (in tiles)
    int nT, nsT;                   // block rows in total, separator block columns
    int ns, nb;                    // separator / boundary unknowns (unpadded; the n_rhs rhs nodes are the last boundary unknowns)
    int idx_off;                   // into idx[]: nT * 64 node ids, -1 = padding, M + d = rhs node of column d
    int pmap_off;                  // into pmap[]: (nT - nsT) * 64 positions in the parent's padded list (-1 = none)
    int parent;
    int child[2];
    int cpos_off[2];               // into cpos[]: nT * 64 boundary-local positions in child c (-1 = none)
    int linv_base;                 // first L(C,C)^-1 tile of this front (nsT tiles)
    int cnt_base;                  // first per-block-column counter of this front (nsT counters)
    int level;
};
__host__ __device__ __forceinline__ long long front_tile(const FrontDesc& f, int R, int C) {
    return f.tile_base + (long long)C * f.nT - (long long)C * (C - 1) / 2 + (R - C);
}

// Pool tiles are stored PADDED: 64 columns of LDT = 68 doubles (element (r, c) at c * LDT + r), the bank-conflict-free layout
// the tensor-core fragment loads want (tile_ops.cuh), so that ONE bulk copy lands an operand ready for dmma_tile — no
// repacking pass, half the shared memory (two CTAs per SM: one computes while the other waits for its operands).
constexpr int TILE_P = NB * LDT;                       // doubles per pool tile
constexpr uint32_t TILE_P_BYTES = TILE_P * 8;
constexpr size_t kNdSmem = 2 * (size_t)TILE_P * sizeof(double);

__device__ __forceinline__ void tma_load_ptile(double* dst_smem, const double* src_gmem, uint64_t* bar) {
    tma_load_bulk(dst_smem, src_gmem, TILE_P_BYTES, bar);
}
__device__ __forceinline__ void regs_from_ptile(double (&acc)[4][4], const double* __restrict__ t, int tm, int tn) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const double2 a = *reinterpret_cast<const double2*>(t + (tn + j) * LDT + tm);
        const double2 b = *reinterpret_cast<const double2*>(t + (tn + j) * LDT + tm + 2);
        acc[0][j] = a.x; acc[1][j] = a.y; acc[2][j] = b.x; acc[3][j] = b.y;
    }
}

struct NdFrontHost {
    int level = 0, parent = -1;
    int child[2] = {-1, -1};
    int r0 = 0, r1 = 0, c0 = 0, c1 = 0;
    std::vector<int> sep, bnd;
};

static int nd_rec(std::vector<NdFrontHost>& F, int r0, int r1, int c0, int c1, int level, int k, int leaf, int m2) {
    const int nr = r1 - r0, nc = c1 - c0;
    const bool can_r = nr >= 3 * k + 2 && nr > leaf, can_c = nc >= 3 * k + 2 && nc > leaf;
    NdFrontHost f;
    f.level = level; f.r0 = r0; f.r1 = r1; f.c0 = c0; f.c1 = c1;
    int a = -1, b = -1;
    if (!(can_r || can_c)) {
        for (int r = r0; r < r1; ++r)
            for (int c = c0; c < c1; ++c) f.sep.push_back(r * m2 + c);
    } else if (can_r && (nr >= nc || !can_c)) {
        const int mid = r0 + (nr - k) / 2;
        for (int r = mid; r < mid + k; ++r)
            for (int c = c0; c < c1; ++c) f.sep.push_back(r * m2 + c);
        a = nd_rec(F, r0, mid, c0, c1, level + 1, k, leaf, m2);
        b = nd_rec(F, mid + k, r1, c0, c1, level + 1, k, leaf, m2);
    } else {
        const int mid = c0 + (nc - k) / 2;
        for (int r = r0; r < r1; ++r)
            for (int c = mid; c < mid + k; ++c) f.sep.push_back(r * m2 + c);
        a = nd_rec(F, r0, r1, c0, mid, level + 1, k, leaf, m2);
        b = nd_rec(F, r0, r1, mid + k, c1, level + 1, k, leaf, m2);
    }
    f.child[0] = a; f.child[1] = b;
    F.push_back(f);
    const int id = (int)F.size() - 1;
    if (a >= 0) { F[a].parent = id; F[b].parent = id; }
    return id;
}

struct NdPlan {
    int m1 = 0, m2 = 0, K = 0, M = 0, R = 1;     // R: right-hand sides (rhs nodes M ... M+R-1)
    int n_fronts = 0, n_levels = 0, root = -1;
    long long n_tiles = 0;         // tiles per pool
    int n_linv = 0, n_cnt = 0;
    std::vector<FrontDesc> fronts;
    std::vector<int> idx, pmap, cpos;
    std::vector<std::vector<int4>> factor_tasks, selinv_tasks, gather_tasks;    // per level
    std::vector<int4> ypass_tasks, all_tasks;
    std::vector<long long> doff, xoff, sigoff;     // xoff[d * M + j]: Sigma'(rhs_d, j)
    std::vector<long long> quad_off;               // [R]: L-pool offsets of the root's update entries (rhs_d, rhs_d)
    // device copies
    FrontDesc* d_fronts = nullptr;
    int *d_idx = nullptr, *d_pmap = nullptr, *d_cpos = nullptr;
    std::vector<int4*> d_factor_tasks, d_selinv_tasks, d_gather_tasks;
    int4 *d_ypass_tasks = nullptr, *d_all_tasks = nullptr;
    long long *d_doff = nullptr, *d_xoff = nullptr, *d_sigoff = nullptr, *d_quad_off = nullptr;
};

constexpr int kNdScalarBlocks = 64;   // slices of the log-determinant sum
constexpr int kNdLeaf = 12;        // regions whose sides are both <= this many grid lines are eliminated as one front

static void nd_build(NdPlan& P, int m1, int m2, int K, int R) {
    P.m1 = m1; P.m2 = m2; P.K = K; P.M = m1 * m2; P.R = R;
    const int M = P.M, RHS = M;
    std::vector<NdFrontHost> F;
    int leaf = kNdLeaf;
    if (const char* e = getenv("ASVGP_ND_LEAF")) leaf = std::max(1, atoi(e));      // tuning knob (tools/nd_leaf_sweep.sh)
    const bool dense = K < 0;      // a dense m1 x m1 matrix (m2 = 1): ONE front holding everything (asvgp_dense_*)
    if (dense) {
        NdFrontHost f;
        f.r1 = m1; f.c1 = 1;
        for (int g = 0; g < M; ++g) f.sep.push_back(g);
        F.push_back(f);
        P.root = 0;
    } else {
        P.root = nd_rec(F, 0, m1, 0, m2, 0, K, leaf, m2);
    }
    P.n_fronts = (int)F.size();
    for (auto& f : F) {            // boundary: ancestors' separator unknowns within K grid lines of the subtree's region
        for (int a = f.parent; a >= 0; a = F[a].parent)
            for (int g : F[a].sep) {
                const int s1 = g / m2, s2 = g % m2;
                if (s1 >= f.r0 - K && s1 <= f.r1 - 1 + K && s2 >= f.c0 - K && s2 <= f.c1 - 1 + K) f.bnd.push_back(g);
            }
        for (int d = 0; d < R; ++d) f.bnd.push_back(RHS + d);
        P.n_levels = std::max(P.n_levels, f.level + 1);
    }
    P.fronts.resize(P.n_fronts);
    std::vector<std::unordered_map<int, int>> pos(P.n_fronts);      // node id -> position in the front's padded list
    long long tiles = 0;
    int linv = 0;
    for (int i = 0; i < P.n_fronts; ++i) {
        FrontDesc& d = P.fronts[i];
        const NdFrontHost& f = F[i];
        d.ns = (int)f.sep.size(); d.nb = (int)f.bnd.size();
        d.nsT = (d.ns + NB - 1) / NB;
        d.nT = d.nsT + (d.nb + NB - 1) / NB;
        d.tile_base = tiles; tiles += (long long)d.nT * (d.nT + 1) / 2;
        d.linv_base = linv; d.cnt_base = linv; linv += d.nsT;
        d.parent = f.parent; d.child[0] = f.child[0]; d.child[1] = f.child[1]; d.level = f.level;
        d.idx_off = (int)P.idx.size();
        P.idx.resize(P.idx.size() + (size_t)d.nT * NB, -1);
        for (int j = 0; j < d.ns; ++j) { P.idx[d.idx_off + j] = f.sep[j]; pos[i][f.sep[j]] = j; }
        for (int j = 0; j < d.nb; ++j) { P.idx[d.idx_off + d.nsT * NB + j] = f.bnd[j]; pos[i][f.bnd[j]] = d.nsT * NB + j; }
    }
    P.n_tiles = tiles; P.n_linv = linv; P.n_cnt = linv;
    for (int i = 0; i < P.n_fronts; ++i) {                          // child -> parent maps and their inverses
        FrontDesc& d = P.fronts[i];
        d.pmap_off = (int)P.pmap.size();
        P.pmap.resize(P.pmap.size() + (size_t)(d.nT - d.nsT) * NB, -1);
        if (d.parent >= 0)
            for (int j = 0; j < d.nb; ++j) P.pmap[d.pmap_off + j] = pos[d.parent].at(F[i].bnd[j]);
        for (int c = 0; c < 2; ++c) {
            d.cpos_off[c] = -1;
            if (d.child[c] < 0) continue;
            d.cpos_off[c] = (int)P.cpos.size();
            P.cpos.resize(P.cpos.size() + (size_t)d.nT * NB, -1);
            const NdFrontHost& ch = F[d.child[c]];
            for (int j = 0; j < (int)ch.bnd.size(); ++j) P.cpos[d.cpos_off[c] + pos[i].at(ch.bnd[j])] = j;
        }
    }
    // task lists.  Factorisation: block column major inside a front (a topological order of its DAG), fronts interleaved so
    // that the chains of diagonal tiles of all fronts advance together.  Selected inverse: block columns descending
    // (counted from each front's last separator column), rows far to near.
    P.factor_tasks.resize(P.n_levels); P.selinv_tasks.resize(P.n_levels); P.gather_tasks.resize(P.n_levels);
    for (int lev = 0; lev < P.n_levels; ++lev) {
        int maxT = 0, maxS = 0;
        for (auto& d : P.fronts) if (d.level == lev) { maxT = std::max(maxT, d.nT); maxS = std::max(maxS, d.nsT); }
        for (int C = 0; C < maxT; ++C)
            for (int i = 0; i < P.n_fronts; ++i) {
                const FrontDesc& d = P.fronts[i];
                if (d.level != lev || C >= d.nT) continue;
                for (int R = C; R < d.nT; ++R) P.factor_tasks[lev].push_back(make_int4(i, R, C, 0));
            }
        for (int back = 0; back < maxS; ++back)
            for (int i = 0; i < P.n_fronts; ++i) {
                const FrontDesc& d = P.fronts[i];
                const int C = d.nsT - 1 - back;
                if (d.level != lev || C < 0) continue;
                for (int R = d.nT - 1; R > C; --R) P.selinv_tasks[lev].push_back(make_int4(i, R, C, 0));
            }
        for (int i = 0; i < P.n_fronts; ++i) {
            const FrontDesc& d = P.fronts[i];
            if (d.level != lev) continue;
            for (int C = d.nsT; C < d.nT; ++C)
                for (int R = C; R < d.nT; ++R) P.gather_tasks[lev].push_back(make_int4(i, R, C, 0));
        }
    }
    for (int i = 0; i < P.n_fronts; ++i) {
        const FrontDesc& d = P.fronts[i];
        for (int C = 0; C < d.nT; ++C)
            for (int R = C; R < d.nT; ++R) {
                if (C < d.nsT) P.ypass_tasks.push_back(make_int4(i, R, C, 0));
                P.all_tasks.push_back(make_int4(i, R, C, 0));
            }
    }
    // element offsets for the scalar / extraction kernels
    std::vector<int> owner(M), opos(M);
    for (int i = 0; i < P.n_fronts; ++i)
        for (int j = 0; j < P.fronts[i].ns; ++j) { owner[F[i].sep[j]] = i; opos[F[i].sep[j]] = j; }
    auto elem = [&](const FrontDesc& d, int prow, int pcol) {       // element (prow, pcol), prow >= pcol, of the front's lower triangle
        return front_tile(d, prow / NB, pcol / NB) * TILE_P + (long long)(pcol % NB) * LDT + prow % NB;
    };
    P.doff.resize(M); P.xoff.resize((size_t)R * M);
    for (int j = 0; j < M; ++j) {
        const FrontDesc& d = P.fronts[owner[j]];
        P.doff[j] = elem(d, opos[j], opos[j]);
        for (int c = 0; c < R; ++c) P.xoff[(size_t)c * M + j] = elem(d, d.nsT * NB + d.nb - R + c, opos[j]);
    }
    {
        const FrontDesc& r = P.fronts[P.root];
        P.quad_off.resize(R);
        for (int c = 0; c < R; ++c) {
            const int p = r.nsT * NB + r.nb - R + c;
            P.quad_off[c] = elem(r, p, p);
        }
    }
    if (dense) return;             // the dense extraction kernel computes its offsets itself (one front)
    const int NS = 2 * K + 1, n_e = (K + 1) * NS;
    P.sigoff.assign((size_t)n_e * M, -1);
    for (int j = 0; j < M; ++j) {
        const int j1 = j / m2, j2 = j % m2;
        for (int d1 = 0; d1 <= K; ++d1)
            for (int d2 = -K; d2 <= K; ++d2) {
                if (d1 == 0 && d2 < 0) continue;
                const int i1 = j1 + d1, i2 = j2 + d2;
                if (i1 >= m1 || i2 < 0 || i2 >= m2) continue;
                const int i = i1 * m2 + i2;
                const int fi = owner[i], fj = owner[j];
                long long off;
                if (fi == fj) {
                    const int hi = std::max(opos[i], opos[j]), lo = std::min(opos[i], opos[j]);
                    off = elem(P.fronts[fi], hi, lo);
                    if (hi / NB == lo / NB) off |= 1LL << 62;          // diagonal tile: average with the mirrored entry
                } else {
                    const bool j_deeper = P.fronts[fj].level > P.fronts[fi].level;
                    const int fd = j_deeper ? fj : fi, nd = j_deeper ? j : i, na = j_deeper ? i : j;
                    off = elem(P.fronts[fd], pos[fd].at(na), opos[nd]);
                }
                P.sigoff[(size_t)(d1 * NS + d2 + K) * M + j] = off;
            }
    }
}

template <class T>
static int nd_upload(T** dst, const std::vector<T>& src) {
    *dst = nullptr;
    if (src.empty()) return kOk;
    ASVGP_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(dst), src.size() * sizeof(T)));
    ASVGP_CUDA_OK(cudaMemcpy(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice));
    return kOk;
}

static std::mutex g_plan_mutex;
static std::map<std::tuple<int, int, int, int, int>, NdPlan*> g_plans;     // (device or -1 for host-only, m1, m2, order, n_rhs)

// host-only plan (sizes, diagnostics); no CUDA calls
static const NdPlan* nd_plan_host(int m1, int m2, int K, int R = 1) {
    std::lock_guard<std::mutex> lock(g_plan_mutex);
    auto key = std::make_tuple(-1, m1, m2, K, R);
    auto it = g_plans.find(key);
    if (it != g_plans.end()) return it->second;
    NdPlan* P = new NdPlan();
    nd_build(*P, m1, m2, K, R);
    g_plans[key] = P;
    return P;
}

static int nd_plan_device(int m1, int m2, int K, int R, const NdPlan** out) {
    int dev = 0;
    ASVGP_CUDA_OK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_plan_mutex);
    auto key = std::make_tuple(dev, m1, m2, K, R);
    auto it = g_plans.find(key);
    if (it != g_plans.end()) { *out = it->second; return kOk; }
    NdPlan* P = new NdPlan();
    nd_build(*P, m1, m2, K, R);
    if (int rc = nd_upload(&P->d_fronts, P->fronts)) return rc;
    if (int rc = nd_upload(&P->d_idx, P->idx)) return rc;
    if (int rc = nd_upload(&P->d_pmap, P->pmap)) return rc;
    if (int rc = nd_upload(&P->d_cpos, P->cpos)) return rc;
    P->d_factor_tasks.resize(P->n_levels); P->d_selinv_tasks.resize(P->n_levels); P->d_gather_tasks.resize(P->n_levels);
    for (int l = 0; l < P->n_levels; ++l) {
        if (int rc = nd_upload(&P->d_factor_tasks[l], P->factor_tasks[l])) return rc;
        if (int rc = nd_upload(&P->d_selinv_tasks[l], P->selinv_tasks[l])) return rc;
        if (int rc = nd_upload(&P->d_gather_tasks[l], P->gather_tasks[l])) return rc;
    }
    if (int rc = nd_upload(&P->d_ypass_tasks, P->ypass_tasks)) return rc;
    if (int rc = nd_upload(&P->d_all_tasks, P->all_tasks)) return rc;
    if (int rc = nd_upload(&P->d_doff, P->doff)) return rc;
    if (int rc = nd_upload(&P->d_xoff, P->xoff)) return rc;
    if (int rc = nd_upload(&P->d_sigoff, P->sigoff)) return rc;
    if (int rc = nd_upload(&P->d_quad_off, P->quad_off)) return rc;
    g_plans[key] = P;
    *out = P;
    return kOk;
}

// Buffer layouts (doubles).  band = [ L tiles | Linv tiles | scalars(8) | flags (ints) ], sig = [ lower tiles | upper tiles ],
// work = [ flags (ints) ]
struct NdLayout {
    long long linv, scal, flags, band_total, n_flag_ints;
    long long sig_upper, sig_total;
    long long work_total, n_work_ints;
};
static NdLayout nd_layout(const NdPlan& P) {
    NdLayout L;
    L.linv = P.n_tiles * TILE_P;
    L.scal = L.linv + (long long)P.n_linv * TILE_P;
    L.flags = L.scal + 8 + kNdScalarBlocks;
    L.n_flag_ints = P.n_tiles + 8;                       // tile flags, abort, first bad pivot, scalar-kernel block counter
    L.band_total = L.flags + (L.n_flag_ints + 1) / 2 + 2;
    L.sig_upper = P.n_tiles * TILE_P;
    L.sig_total = 2 * L.sig_upper;
    L.n_work_ints = P.n_tiles + P.n_cnt + 8;             // tile flags, per-block-column counters, abort
    L.work_total = (L.n_work_ints + 1) / 2 + 2;
    return L;
}

// ---------------------------------------------------------------------------------------------------------------------
// assembly: entries of P (+ right-hand side row) of every front, one fully parallel launch; the children's update matrices
// are added by the children's own factorisation tasks (scatter_to_parent)
// ---------------------------------------------------------------------------------------------------------------------
// Slot s of a batch (blockIdx.y) assembles K1 + s k1_stride, K2 + s k2_stride and sigma2[s] into Lpool + s band_stride; Gs
// and b are shared.  The single calls are the one-slot case.
struct NdAssembleArgs {
    const FrontDesc* fronts; const int4* tasks; int n_tasks;
    const int* idx;
    const double *K1, *K2, *Gs, *b;
    int m1, m2, K, M;
    double* Lpool;
    const double* dense;           // non-null: the matrix itself, M x M row-major (lower triangle read), instead of K1, K2, Gs
    long long band_stride, k1_stride, k2_stride;
    double sigma2[ASVGP_MAX_BATCH];
};

__device__ __forceinline__ double nd_band_sym(const double* B, int m, int K, int i, int j) {
    const int d = i > j ? i - j : j - i;
    return d <= K ? __ldg(B + (long long)d * m + (i < j ? i : j)) : 0.0;
}

// A'(gi, gj): gi, gj grid unknowns or rhs nodes (id M + d: A'(g, rhs_d) = b[d M + g], A'(rhs_d, rhs_e) = 0).  Same roundings as
// the reference's `Kuu + KufKfu / sigma2`.
__device__ __forceinline__ double nd_entry(const NdAssembleArgs& a, const double* K1, const double* K2, double sigma2, int gi, int gj) {
    if (gi >= a.M || gj >= a.M) {
        if (gi >= a.M && gj >= a.M) return 0.0;
        return gi >= a.M ? __ldg(a.b + (long long)(gi - a.M) * a.M + gj) : __ldg(a.b + (long long)(gj - a.M) * a.M + gi);
    }
    if (a.dense != nullptr) return __ldg(a.dense + (long long)max(gi, gj) * a.M + min(gi, gj));
    const int i1 = gi / a.m2, i2 = gi % a.m2, j1 = gj / a.m2, j2 = gj % a.m2;
    int d1 = i1 - j1, d2 = i2 - j2;
    int col = gj;
    if (d1 < 0 || (d1 == 0 && d2 < 0)) { d1 = -d1; d2 = -d2; col = gi; }
    if (d1 > a.K || d2 > a.K || d2 < -a.K) return 0.0;
    const double kv = __dmul_rn(nd_band_sym(K1, a.m1, a.K, i1, j1), nd_band_sym(K2, a.m2, a.K, i2, j2));
    const double g = __ldg(a.Gs + (long long)(d1 * (2 * a.K + 1) + d2 + a.K) * a.M + col);
    return __dadd_rn(kv, __ddiv_rn(g, sigma2));
}

__global__ void __launch_bounds__(256) nd_assemble_kernel(const __grid_constant__ NdAssembleArgs a) {
    const int slot = blockIdx.y;
    const double* K1 = a.K1 + slot * a.k1_stride;
    const double* K2 = a.K2 + slot * a.k2_stride;
    const double sigma2 = a.sigma2[slot];
    double* Lpool = a.Lpool + slot * a.band_stride;
    for (int t = blockIdx.x; t < a.n_tasks; t += gridDim.x) {
        const int4 tk = a.tasks[t];
        const FrontDesc f = a.fronts[tk.x];
        const int R = tk.y, C = tk.z;
        double* tile = Lpool + front_tile(f, R, C) * TILE_P;
        const int* idx = a.idx + f.idx_off;
        if (C >= f.nsT && f.child[0] < 0) continue;          // trailing tiles of a leaf front start from zero: never read
        for (int e = threadIdx.x; e < TILE; e += blockDim.x) {
            const int r = e % NB, c = e / NB;
            const int I = R * NB + r, J = C * NB + c;
            const int gi = idx[I], gj = idx[J];
            double v;
            if (gi < 0 || gj < 0) v = (I == J && C < f.nsT) ? 1.0 : 0.0;
            else v = (C < f.nsT) ? nd_entry(a, K1, K2, sigma2, gi, gj) : 0.0;
            tile[c * LDT + r] = v;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// factorisation of all fronts of one level
// ---------------------------------------------------------------------------------------------------------------------
// A batch of n_slots settings: combined task t is task t / n_slots of slot t % n_slots (task-major, so every slot keeps its own
// task order and a task still waits only on tasks dealt before it), and slot s owns the band buffer at s band_stride doubles.
struct NdFactorArgs {
    const FrontDesc* fronts; const int4* tasks; int n_tasks;
    const int *idx, *pmap;
    double* Lpool; double* linv;
    int* ready;         // [n_tiles] + abort at [n_tiles], first bad pivot (node id + 1) at [n_tiles + 1]
    long long n_tiles;
    int n_slots;
    long long band_stride;
};

// Extend-add, from the child's side: this thread's 4 x 4 block of the update tile (R, C) of front f (R >= C >= nsT) is added
// into the parent's front (fp64 REDs: the two children of a parent add into the same entries; the parent was assembled before
// any factorisation kernel ran and is factorised by a later launch).  The parent stores its lower triangle, with FULL diagonal
// tiles; the child's diagonal update tiles are full too, so only their lower triangle is sent.
__device__ __forceinline__ void scatter_to_parent(const double (&acc)[4][4], const NdFactorArgs& a, double* Lpool, const FrontDesc& f,
                                                  int R, int C, int tm, int tn) {
    const FrontDesc p = a.fronts[f.parent];
    const int* pm = a.pmap + f.pmap_off;
    int pr[4], pc[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { pr[i] = __ldg(pm + (R - f.nsT) * NB + tm + i); pc[i] = __ldg(pm + (C - f.nsT) * NB + tn + i); }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (pr[i] < 0 || pc[j] < 0 || (R == C && tm + i < tn + j)) continue;
            const int hi = max(pr[i], pc[j]), lo = min(pr[i], pc[j]);
            double* t = Lpool + front_tile(p, hi / NB, lo / NB) * TILE_P;
            atomicAdd(t + (lo % NB) * LDT + hi % NB, acc[i][j]);
            if (hi / NB == lo / NB && hi != lo) atomicAdd(t + (hi % NB) * LDT + lo % NB, acc[i][j]);
        }
}

__global__ void __launch_bounds__(kTdThreads, 2) nd_factor_kernel(NdFactorArgs a) {
    extern __shared__ __align__(128) unsigned char td_smem[];
    double* const pA = reinterpret_cast<double*>(td_smem);                 // landing buffers of the two operands of a product
    double* const pB = pA + TILE_P;
    __shared__ __align__(8) uint64_t full;
    __shared__ int s_bad;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tm = (tid & 15) * 4, tn = (tid >> 4) * 4;
    if (tid == 0) mbar_init(&full, 1);
    fence_proxy_async();
    __syncthreads();
    uint32_t phase = 0;

    for (int t = blockIdx.x; t < a.n_tasks * a.n_slots; t += gridDim.x) {
        const int slot = t % a.n_slots;
        const int4 tk = a.tasks[t / a.n_slots];
        double* const Lpool = a.Lpool + slot * a.band_stride;
        double* const linv = a.linv + slot * a.band_stride;
        int* const ready = a.ready + 2 * slot * a.band_stride;
        int* const abort_flag = ready + a.n_tiles;
        const FrontDesc f = a.fronts[tk.x];
        const int R = tk.y, C = tk.z;
        const bool diag = R == C;
        double* my_tile = Lpool + front_tile(f, R, C) * TILE_P;
        const int nJ = min(C, f.nsT);

        auto issue = [&](int J) {                    // thread 0: wait for the operand tiles, then fetch them by TMA
            const long long tR = front_tile(f, R, J), tC = front_tile(f, C, J);
            wait_flag(ready + tR, 1, abort_flag);
            if (!diag) wait_flag(ready + tC, 1, abort_flag);
            fence_proxy_async();
            mbar_expect_tx(&full, diag ? TILE_P_BYTES : 2 * TILE_P_BYTES);
            tma_load_ptile(pA, Lpool + tR * TILE_P, &full);
            if (!diag) tma_load_ptile(pB, Lpool + tC * TILE_P, &full);
        };
        if (tid == 0 && nJ > 0) issue(0);
        double acc[4][4];
        if (C >= f.nsT && f.child[0] < 0) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
        } else {
            regs_from_ptile(acc, my_tile, tm, tn);
        }
        if (nJ > 0) {
            double cf[8][2] = {};                    // sum_J L(R,J) L(C,J)^T as tensor-core fragments
            for (int q = 0; q < nJ; ++q) {
                mbar_wait(&full, phase);
                phase ^= 1u;
                dmma_tile(cf, pA, diag ? pA : pB, warp, lane);
                __syncthreads();
                if (q + 1 < nJ && tid == 0) issue(q + 1);
            }
            frags_subtract(acc, cf, pA, warp, lane, tm, tn);
        }

        if (C >= f.nsT) {
            // ---- trailing tile: this front's update matrix, added straight into the parent's front --------------------------
            if (f.parent >= 0) scatter_to_parent(acc, a, Lpool, f, R, C, tm, tn);
            else regs_to_tile_ld<LDT>(acc, my_tile, tm, tn);     // root: entry (rhs, rhs) = -||y||^2
        } else if (diag) {
            // ---- diagonal tile: Cholesky + inverse in registers ---------------------------------------------------------------
            double V[4][4];
            double* s11 = pA;                        // [16] l + [4] 1/l_cc (+ padding)
            double* spanel = pA + 32;                // [4][64] panel, transposed
            double* swrow = pA + 32 + 4 * NB;        // [4][64]
            if (tid == 0) s_bad = -1;
            __syncthreads();
            potrf_regs(acc, V, tm, tn, s11, spanel, swrow, &s_bad, nullptr);
            __syncthreads();
            const int first_bad = s_bad;
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (tm + i < tn + j) { acc[i][j] = 0.0; V[i][j] = 0.0; }
                }
            regs_to_tile_ld<LDT>(V, linv + (long long)(f.linv_base + C) * TILE_P, tm, tn);
            regs_to_tile_ld<LDT>(acc, my_tile, tm, tn);
            __threadfence();
            __syncthreads();
            if (tid == 0) {
                st_release(ready + front_tile(f, C, C), 1);
                if (first_bad >= 0) atomicMin(ready + a.n_tiles + 1, a.idx[f.idx_off + C * NB + first_bad] + 1);
            }
        } else {
            // ---- sub-diagonal tile: L(R,C) = A L(C,C)^-T -------------------------------------------------------------------------
            if (tid == 0) {
                wait_flag(ready + front_tile(f, C, C), 1, abort_flag);
                fence_proxy_async();
                mbar_expect_tx(&full, TILE_P_BYTES);
                tma_load_ptile(pB, linv + (long long)(f.linv_base + C) * TILE_P, &full);
            }
            regs_to_tile_ld<LDT>(acc, pA, tm, tn);   // A(m, k) at [k*LDT + m]
            __syncthreads();
            mbar_wait(&full, phase);
            phase ^= 1u;
            double L[4][4] = {};
            {
                double cf[8][2] = {};
                dmma_tile(cf, pA, pB, warp, lane);                  // L[m][n] = sum_k A[m][k] Linv[n][k]
                __syncthreads();
                frags_subtract(L, cf, pA, warp, lane, tm, tn);
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) L[i][j] = -L[i][j];
            }
            regs_to_tile_ld<LDT>(L, my_tile, tm, tn);
            __threadfence();
            __syncthreads();
            if (tid == 0) st_release(ready + front_tile(f, R, C), 1);
        }
        __syncthreads();
    }
}

// log|P| = 2 sum log L_jj (deterministic: fixed slices, tree reductions, the last block to finish adds the slices in order),
// ||y_d||^2 = -(root update entry (rhs_d, rhs_d)), info, and tau.  scal_out[0] = log|P|, scal_out[q_slot + d] = ||y_d||^2,
// scal_out[info_slot] = info.  Slot blockIdx.y of a batch: its band buffer at blockIdx.y band_stride doubles (Lpool, ready and
// scal_keep move with it), its scalars at scal_out + blockIdx.y scal_stride.
__global__ void __launch_bounds__(256) nd_scalars_kernel(const long long* __restrict__ doff, int M, const double* __restrict__ Lpool,
                                                         const long long* __restrict__ quad_off, int R, int q_slot, int info_slot,
                                                         int* __restrict__ ready, long long n_tiles,
                                                         double* __restrict__ scal_out, double* __restrict__ scal_keep,
                                                         long long band_stride, int scal_stride) {
    __shared__ double s[256];
    Lpool += blockIdx.y * band_stride;
    ready += 2 * blockIdx.y * band_stride;
    scal_keep += blockIdx.y * band_stride;
    scal_out += blockIdx.y * scal_stride;
    __shared__ bool last;
    double acc = 0.0;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < M; j += gridDim.x * blockDim.x) acc += log(__ldcg(Lpool + doff[j]));
    s[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        scal_keep[8 + blockIdx.x] = s[0];
        __threadfence();
        last = atomicAdd(ready + n_tiles + 2, 1) == (int)gridDim.x - 1;
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int bk = 0; bk < (int)gridDim.x; ++bk) tot += __ldcg(scal_keep + 8 + bk);
        const int aborted = ready[n_tiles], bad = ready[n_tiles + 1];
        scal_out[0] = 2.0 * tot;
        double quad = 0.0;
        for (int d = 0; d < R; ++d) {
            const double q = -__ldcg(Lpool + quad_off[d]);
            scal_out[q_slot + d] = q;
            quad = d == 0 ? q : quad + q;
        }
        scal_out[info_slot] = aborted ? -1.0 : (bad != kNoBadPivot ? (double)bad : 0.0);
        scal_keep[0] = quad;
        scal_keep[1] = 9.5367431640625e-07 / (1.0 + quad);        // tau = 2^-20 / (1 + sum_d ||y_d||^2)
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// selected inverse
// ---------------------------------------------------------------------------------------------------------------------
// Pre-pass over every tile (R, C), C < nsT, of every front, fully parallel: off-diagonal tiles become Y^T
// (Y = L(R,C) L(C,C)^-1, stored transposed so that it is a plain operand later), diagonal tiles seed
// Sigma(C,C) = L(C,C)^-T L(C,C)^-1.  Slot blockIdx.y of a batch: Lpool, linv + blockIdx.y band_stride, sig_lower + blockIdx.y sig_stride.
__global__ void __launch_bounds__(kTdThreads) nd_ypass_kernel(const FrontDesc* __restrict__ fronts, const int4* __restrict__ tasks,
                                                              int n_tasks, double* __restrict__ Lpool, const double* __restrict__ linv,
                                                              double* __restrict__ sig_lower, long long band_stride, long long sig_stride) {
    extern __shared__ __align__(16) unsigned char yp_smem[];
    Lpool += blockIdx.y * band_stride;
    linv += blockIdx.y * band_stride;
    sig_lower += blockIdx.y * sig_stride;
    double* pL = reinterpret_cast<double*>(yp_smem);         // L tile as the A operand: L[m][k] at [k*LDT + m]
    double* pI = pL + TILE_P;                                // Linv transposed: Linv[k][n] at [k*LDT + n]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int t = blockIdx.x; t < n_tasks; t += gridDim.x) {
        const int4 tk = tasks[t];
        const FrontDesc f = fronts[tk.x];
        const int R = tk.y, C = tk.z;
        const double* Li = linv + (long long)(f.linv_base + C) * TILE_P;
        double* T = Lpool + front_tile(f, R, C) * TILE_P;
        __syncthreads();
        for (int e = tid; e < TILE; e += kTdThreads) {
            const int r = e % NB, c = e / NB;
            pI[r * LDT + c] = __ldcg(Li + c * LDT + r);       // Linv[r][c]
            if (R != C) pL[c * LDT + r] = __ldcg(T + c * LDT + r);
        }
        __syncthreads();
        double cf[8][2] = {};
        // diagonal: S0[m][n] = sum_k Linv[k][m] Linv[k][n];  off-diagonal: Y[m][n] = sum_k L[m][k] Linv[k][n]
        dmma_tile(cf, R == C ? pI : pL, pI, warp, lane);
        double* out = (R == C) ? sig_lower + front_tile(f, C, C) * TILE_P : T;     // Y is stored transposed (row m contiguous), in place
        const int m = warp * 8 + (lane >> 2), n0 = (lane & 3) * 2;
#pragma unroll
        for (int cb = 0; cb < 8; ++cb)
            *reinterpret_cast<double2*>(out + m * LDT + cb * 8 + n0) = make_double2(cf[cb][0], cf[cb][1]);
    }
}

// Sigma on the boundary block of every front of a level, from the parent's Sigma (the root's boundary is the rhs nodes
// alone: Sigma'(rhs, rhs) = tau I).  Lower tiles and their transposes.
struct NdGatherArgs {
    const FrontDesc* fronts; const int4* tasks; int n_tasks;
    const int* pmap;
    double *sig_lower, *sig_upper;
    const double* scal_keep;        // [1] = tau
    int n_rhs;
    long long band_stride, sig_stride;      // slot blockIdx.y: scal_keep + y band_stride, sig_* + y sig_stride
};
__global__ void __launch_bounds__(256) nd_gather_kernel(NdGatherArgs a) {
    __shared__ double s_t[NB][NB + 1];
    a.sig_lower += blockIdx.y * a.sig_stride;
    a.sig_upper += blockIdx.y * a.sig_stride;
    a.scal_keep += blockIdx.y * a.band_stride;
    for (int t = blockIdx.x; t < a.n_tasks; t += gridDim.x) {
        const int4 tk = a.tasks[t];
        const FrontDesc f = a.fronts[tk.x];
        const int R = tk.y, C = tk.z;
        const long long me = front_tile(f, R, C);
        const int* pm = a.pmap + f.pmap_off;
        FrontDesc p;
        if (f.parent >= 0) p = a.fronts[f.parent];
        const int rhs_pos = f.nb - a.n_rhs;                              // boundary-local position of the first rhs node
        __syncthreads();
        for (int e = threadIdx.x; e < TILE; e += blockDim.x) {
            const int r = e % NB, c = e / NB;
            const int I = (R - f.nsT) * NB + r, J = (C - f.nsT) * NB + c;
            double v = 0.0;
            if (f.parent < 0) {
                v = (I == J && I >= rhs_pos && I < f.nb) ? a.scal_keep[1] : 0.0;
            } else {
                int pa = pm[I], pb = pm[J];
                if (pa >= 0 && pb >= 0) {
                    if (pa < pb) { const int s = pa; pa = pb; pb = s; }
                    const double* src = a.sig_lower + front_tile(p, pa / NB, pb / NB) * TILE_P;
                    int rr = pa % NB, cc = pb % NB;
                    if (pa / NB == pb / NB && rr < cc) { const int s = rr; rr = cc; cc = s; }   // diagonal tile of the parent: its lower triangle
                    v = __ldcg(src + cc * LDT + rr);
                }
            }
            a.sig_lower[me * TILE_P + c * LDT + r] = v;
            s_t[r][c] = v;
        }
        __syncthreads();
        for (int e = threadIdx.x; e < TILE; e += blockDim.x) a.sig_upper[me * TILE_P + (e / NB) * LDT + e % NB] = s_t[e / NB][e % NB];   // (r,c) <- (c,r)
    }
}

struct NdSelArgs {
    const FrontDesc* fronts; const int4* tasks; int n_tasks;
    const double* Lpool;    // Y^T tiles (off-diagonal) from the pre-pass
    double* sig_lower;      // Sigma(R, C) tiles, R >= C
    double* sig_upper;      // their transposes
    int* sready;            // [n_tiles] tile flags, [n_cnt] per-block-column counters, abort
    long long n_tiles;
    int n_cnt;
    int n_slots;            // tasks dealt task-major over the slots, as in nd_factor_kernel
    long long band_stride, sig_stride, work_stride;     // doubles between the slots' buffers
};

// A diagonal Sigma tile is symmetric only up to rounding (a sum of REDs of termwise unsymmetric products): the operand handed
// to the tensor cores is 0.5 (S + S^T), in place in shared memory (see repack_padded_sym in tile_ops.cuh for why).
__device__ __forceinline__ void symmetrise_ptile(double* __restrict__ s, int tid) {
    const int c = tid & (NB - 1), g = tid >> 6;
    double v[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const int r = (c + g * 16 + j) & (NB - 1);
        v[j] = 0.5 * (s[c * LDT + r] + s[r * LDT + c]);
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 16; ++j) s[c * LDT + ((c + g * 16 + j) & (NB - 1))] = v[j];
}

// kBatched = false is the single-setting kernel (one slot; the kernel sits at its 128-register cap, and the slot arithmetic of
// the batched instance would make it spill).
template <bool kBatched>
__global__ void __launch_bounds__(kTdThreads, 2) nd_selinv_kernel(NdSelArgs a) {
    extern __shared__ __align__(128) unsigned char td_smem[];
    double* const pA = reinterpret_cast<double*>(td_smem);
    double* const pB = pA + TILE_P;
    __shared__ __align__(8) uint64_t full;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tm = (tid & 15) * 4, tn = (tid >> 4) * 4;
    if (tid == 0) mbar_init(&full, 1);
    fence_proxy_async();
    __syncthreads();
    uint32_t phase = 0;

    for (int t = blockIdx.x; t < a.n_tasks * (kBatched ? a.n_slots : 1); t += gridDim.x) {
        const int slot = kBatched ? t % a.n_slots : 0;
        const int4 tk = a.tasks[kBatched ? t / a.n_slots : t];
        const double* const Lpool = a.Lpool + slot * a.band_stride;
        double* const sig_lower = a.sig_lower + slot * a.sig_stride;
        double* const sig_upper = a.sig_upper + slot * a.sig_stride;
        int* const sready = a.sready + 2 * slot * a.work_stride;
        int* const cnt = sready + a.n_tiles;
        int* const abort_flag = cnt + a.n_cnt;
        const FrontDesc f = a.fronts[tk.x];
        const int R = tk.y, C = tk.z;                // R > C, C < nsT
        const int Kmax = f.nT - 1, nK = Kmax - C;
        auto issue = [&](int K) {                    // A = Sigma(R, K), B = Y(K, C)^T
            const double* src;
            const int* flag = nullptr;
            int want = 1;
            if (K == R) {
                src = sig_lower + front_tile(f, R, R) * TILE_P;
                if (R < f.nsT) { flag = cnt + f.cnt_base + R; want = f.nT - 1 - R; }      // all shares in
            } else if (K < R) {
                src = sig_lower + front_tile(f, R, K) * TILE_P;
                if (K < f.nsT) flag = sready + front_tile(f, R, K);
            } else {
                src = sig_upper + front_tile(f, K, R) * TILE_P;
                if (R < f.nsT) flag = sready + front_tile(f, K, R);
            }
            // the Y^T operand is there since the pre-pass: it is requested before the wait, only Sigma(R,K) after it
            mbar_expect_tx(&full, 2 * TILE_P_BYTES);
            tma_load_ptile(pB, Lpool + front_tile(f, K, C) * TILE_P, &full);
            if (flag != nullptr) wait_flag(flag, want, abort_flag);
            fence_proxy_async();
            tma_load_ptile(pA, src, &full);
        };
        double acc[4][4] = {};
        double cf[8][2] = {};                        // sum_K Sigma(R,K) Y(K,C) as tensor-core fragments
        if (tid == 0) issue(Kmax);
        for (int q = 0; q < nK; ++q) {
            mbar_wait(&full, phase);
            phase ^= 1u;
            if (Kmax - q == R) { symmetrise_ptile(pA, tid); __syncthreads(); }
            dmma_tile(cf, pA, pB, warp, lane);
            __syncthreads();
            if (tid == 0) {
                if (q + 1 < nK) {
                    issue(Kmax - q - 1);
                } else {
                    // after the last product: fetch this tile's own Y^T for the diagonal contribution below
                    mbar_expect_tx(&full, TILE_P_BYTES);
                    tma_load_ptile(pB, Lpool + front_tile(f, R, C) * TILE_P, &full);
                }
            }
        }
        frags_subtract(acc, cf, pA, warp, lane, tm, tn);                // acc = -sum_K Sigma(R,K) Y(K,C)
        const long long me = front_tile(f, R, C);
        regs_to_tile_ld<LDT>(acc, sig_lower + me * TILE_P, tm, tn);
        regs_to_tile_t_ld<LDT>(acc, pA, tm, tn);         // T[m][a] at [m*LDT + a]  ==  A'(a, k=m) at [k*LDT + a]
        __syncthreads();
        {
            double* up = sig_upper + me * TILE_P;
#pragma unroll
            for (int idx = tid; idx < TILE / 2; idx += kTdThreads) {
                const int c = idx >> 5, r = (idx & 31) * 2;
                *reinterpret_cast<double2*>(up + c * LDT + r) = *reinterpret_cast<const double2*>(pA + c * LDT + r);
            }
        }
        __threadfence();
        __syncthreads();
        if (tid == 0) st_release(sready + me, 1);
        mbar_wait(&full, phase);
        phase ^= 1u;
        {
            // D[a][b] = sum_m T[m][a] Y[m][b]: this tile's share of Sigma(C,C), added as REDs
            double D[8][2] = {};
            dmma_tile(D, pA, pB, warp, lane);
            double* Sd = sig_lower + front_tile(f, C, C) * TILE_P;
            const int row = warp * 8 + (lane >> 2), col = (lane & 3) * 2;
#pragma unroll
            for (int cb = 0; cb < 8; ++cb) {
                atomicAdd(Sd + (cb * 8 + col) * LDT + row, -D[cb][0]);
                atomicAdd(Sd + (cb * 8 + col + 1) * LDT + row, -D[cb][1]);
            }
        }
        __threadfence();
        __syncthreads();
        if (tid == 0) red_release_add(cnt + f.cnt_base + C, 1);
    }
}

// x[d M + j] = x_d,j = -Sigma'(rhs_d, j) / tau  (t < R M)
// Slot blockIdx.y of a batch: sig_lower + y sig_stride, scal_keep + y band_stride, abort_flag + 2 y work_stride, x + y RM.
__global__ void __launch_bounds__(256) nd_x_kernel(const long long* __restrict__ xoff, int RM, const double* __restrict__ sig_lower,
                                                   const double* __restrict__ scal_keep, const int* __restrict__ abort_flag,
                                                   double* __restrict__ x, long long band_stride, long long sig_stride,
                                                   long long work_stride) {
    sig_lower += blockIdx.y * sig_stride;
    scal_keep += blockIdx.y * band_stride;
    abort_flag += 2 * blockIdx.y * work_stride;
    x += (long long)blockIdx.y * RM;
    const double inv_tau = -1.0 / scal_keep[1];
    const bool aborted = *abort_flag != 0;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < RM; j += gridDim.x * blockDim.x)
        x[j] = aborted ? nan("") : __ldcg(sig_lower + xoff[j]) * inv_tau;
}

// tau sum_d x_d,i x_d,j for R > 1 right-hand sides
__device__ __forceinline__ double nd_rank_correction(const double* __restrict__ x, long long M, int R, double tau, long long i,
                                                     long long j) {
    double c = tau * x[i] * x[j];
    for (int d = 1; d < R; ++d) c += tau * x[d * M + i] * x[d * M + j];
    return c;
}

// stencil entries of P^-1 = Sigma' - tau sum_d x_d x_d^T.  Slot blockIdx.y of a batch: as nd_x_kernel, out + y total.
__global__ void __launch_bounds__(256) nd_stencil_kernel(const long long* __restrict__ sigoff, int m1, int m2, int K, int R,
                                                         const double* __restrict__ sig_lower, const double* __restrict__ x,
                                                         const double* __restrict__ scal_keep, const int* __restrict__ abort_flag,
                                                         double* __restrict__ out, long long band_stride, long long sig_stride,
                                                         long long work_stride) {
    const int NS = 2 * K + 1, n_e = (K + 1) * NS;
    const long long M = (long long)m1 * m2, total = M * n_e;
    sig_lower += blockIdx.y * sig_stride;
    scal_keep += blockIdx.y * band_stride;
    abort_flag += 2 * blockIdx.y * work_stride;
    x += blockIdx.y * M * R;
    out += blockIdx.y * total;
    const double tau = scal_keep[1];
    const bool aborted = *abort_flag != 0;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        long long off = sigoff[t];
        double v = 0.0;
        if (off >= 0) {
            const bool diag_tile = (off >> 62) & 1;
            off &= ~(1LL << 62);
            v = __ldcg(sig_lower + off);
            if (diag_tile) {
                const int e = (int)(off % TILE_P);                      // c * LDT + r inside the tile
                v = 0.5 * (v + __ldcg(sig_lower + (off - e) + (e % LDT) * LDT + e / LDT));
            }
            const int ee = (int)(t / M);
            const long long j = t % M;
            const long long i = j + (long long)(ee / NS) * m2 + (ee % NS - K);
            if (R == 1) v -= tau * x[i] * x[j];          // the single-rhs expression as it was (same contraction, same bits)
            else v -= nd_rank_correction(x, M, R, tau, i, j);
        }
        out[t] = aborted ? nan("") : v;
    }
}

template <class Kernel>
static int nd_launch_persistent(Kernel kernel, void* args, int n_tasks, cudaStream_t st) {
    int dev = 0, sms = 0, per_sm = 0;
    ASVGP_CUDA_OK(cudaGetDevice(&dev));
    ASVGP_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    ASVGP_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kNdSmem));
    ASVGP_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kTdThreads, kNdSmem));
    if (per_sm < 1) {
        set_last_error("front kernel does not fit on an SM (%zu bytes of shared memory)", kNdSmem);
        return kCudaError;
    }
    const int grid = std::max(1, std::min(sms * std::min(per_sm, 2), n_tasks));     // all CTAs co-resident (they wait on each other)
    void* params[] = {args};
    ASVGP_CUDA_OK(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(kernel), dim3(grid), dim3(kTdThreads), params, kNdSmem, st));
    ASVGP_LAUNCHED();
    return kOk;
}

}  // namespace asvgp

using namespace asvgp;

#define ND_CHECK_ARGS(name)                                                                                              \
    ASVGP_REQUIRE(m1 > 0 && m2 > 0 && order >= 1 && order <= kMaxOrder, name ": m=%d,%d order=%d", m1, m2, order)

extern "C" int64_t asvgp_kron_band_doubles(int m1, int m2, int order) {
    if (m1 <= 0 || m2 <= 0 || order < 1 || order > kMaxOrder) return -1;
    return nd_layout(*nd_plan_host(m1, m2, order)).band_total;
}
extern "C" int64_t asvgp_kron_sig_doubles(int m1, int m2, int order) {
    if (m1 <= 0 || m2 <= 0 || order < 1 || order > kMaxOrder) return -1;
    return nd_layout(*nd_plan_host(m1, m2, order)).sig_total;
}
extern "C" int64_t asvgp_kron_work_doubles(int m1, int m2, int order) {
    if (m1 <= 0 || m2 <= 0 || order < 1 || order > kMaxOrder) return -1;
    return nd_layout(*nd_plan_host(m1, m2, order)).work_total;
}
extern "C" int64_t asvgp_kron_rhs_doubles(int m1, int m2, int order) {
    if (m1 <= 0 || m2 <= 0 || order < 1 || order > kMaxOrder) return -1;
    return (int64_t)m1 * m2;
}

#define ND_CHECK_RHS(name)                                                                                               \
    ASVGP_REQUIRE(n_rhs >= 1 && n_rhs <= ASVGP_MAX_RHS, name ": n_rhs=%d (1 ... %d right-hand sides)", n_rhs, ASVGP_MAX_RHS)

static void nd_sizes(const NdPlan& P, int64_t* h_sizes) {
    const NdLayout L = nd_layout(P);
    h_sizes[0] = L.band_total; h_sizes[1] = L.sig_total; h_sizes[2] = L.work_total; h_sizes[3] = (int64_t)P.M * P.R;
}

extern "C" int asvgp_kron_doubles_multi(int m1, int m2, int order, int n_rhs, int64_t* h_sizes) {
    ND_CHECK_ARGS("kron_doubles_multi");
    ND_CHECK_RHS("kron_doubles_multi");
    nd_sizes(*nd_plan_host(m1, m2, order, n_rhs), h_sizes);
    return kOk;
}

// Diagnostics / tests: out[0..7] = fronts, levels, tiles per pool, separator block columns, sum of separator sizes along the
// longest root-to-leaf path (the dependency chain, in columns), the same in block columns, largest front (unknowns), flops.
// idx_out (may be NULL): for every front, level, ns, nb, then the ns + nb node ids (rhs nodes = m1*m2 ... m1*m2+n_rhs-1);
// returns the number of ints that takes.
static int64_t nd_plan_info(int m1, int m2, int order, int n_rhs, double* out, int32_t* idx_out, int64_t idx_capacity);

extern "C" int64_t asvgp_kron_plan_info(int m1, int m2, int order, double* out, int32_t* idx_out, int64_t idx_capacity) {
    if (m1 <= 0 || m2 <= 0 || order < 1 || order > kMaxOrder) return -1;
    return nd_plan_info(m1, m2, order, 1, out, idx_out, idx_capacity);
}

extern "C" int64_t asvgp_kron_plan_info_multi(int m1, int m2, int order, int n_rhs, double* out, int32_t* idx_out,
                                              int64_t idx_capacity) {
    if (m1 <= 0 || m2 <= 0 || order < 1 || order > kMaxOrder) {
        set_last_error("kron_plan_info_multi: m=%d,%d order=%d", m1, m2, order);
        return -1;
    }
    if (n_rhs < 1 || n_rhs > ASVGP_MAX_RHS) {
        set_last_error("kron_plan_info_multi: n_rhs=%d (1 ... %d right-hand sides)", n_rhs, ASVGP_MAX_RHS);
        return -1;
    }
    return nd_plan_info(m1, m2, order, n_rhs, out, idx_out, idx_capacity);
}

static int64_t nd_plan_info(int m1, int m2, int order, int n_rhs, double* out, int32_t* idx_out, int64_t idx_capacity) {
    const NdPlan& P = *nd_plan_host(m1, m2, order, n_rhs);
    std::vector<long long> chain(P.n_fronts, 0), chainT(P.n_fronts, 0);
    double flops = 0.0;
    long long best = 0, bestT = 0;
    int largest = 0;
    for (int i = P.n_fronts - 1; i >= 0; --i) {                  // parents come after children: walk from the root down
        const FrontDesc& d = P.fronts[i];
        chain[i] = d.ns + (d.parent >= 0 ? chain[d.parent] : 0);
        chainT[i] = d.nsT + (d.parent >= 0 ? chainT[d.parent] : 0);
        best = std::max(best, chain[i]); bestT = std::max(bestT, chainT[i]);
        largest = std::max(largest, d.ns + d.nb);
        flops += (double)d.ns * (d.ns + d.nb) * (d.ns + d.nb);
    }
    if (out != nullptr) {
        out[0] = P.n_fronts; out[1] = P.n_levels; out[2] = (double)P.n_tiles; out[3] = P.n_linv;
        out[4] = (double)best; out[5] = (double)bestT; out[6] = largest; out[7] = flops;
    }
    int64_t need = 0;
    for (const FrontDesc& d : P.fronts) need += 3 + d.ns + d.nb;
    if (idx_out != nullptr && idx_capacity >= need) {
        int64_t w = 0;
        for (const FrontDesc& d : P.fronts) {
            idx_out[w++] = d.level; idx_out[w++] = d.ns; idx_out[w++] = d.nb;
            for (int j = 0; j < d.ns; ++j) idx_out[w++] = P.idx[d.idx_off + j];
            for (int j = 0; j < d.nb; ++j) idx_out[w++] = P.idx[d.idx_off + d.nsT * NB + j];
        }
    }
    return need;
}


// ---- shared bodies of the Kronecker and the dense entry points -----------------------------------------------------------------
// A batch of B settings on one plan: slot s owns band + s band, sig_band + s sig, work + s work (strides in doubles, 0 for the
// single calls), its scalars at scal + s scal_stride and its x at x_out + s n_rhs M.
struct NdBatch {
    int B = 1;
    long long band = 0, sig = 0, work = 0;
    int scal = 0;
};
// CTAs per slot of the fully parallel kernels: the single call's `cap`, shared out over the slots
static int nd_grid_x(long long n, int cap, int B) { return (int)std::max<long long>(1, std::min<long long>(n, (cap + B - 1) / B)); }

// multi = false: scal = { log|P|, Q, info } (single-rhs layout); true: scal = { log|P|, info, Q_1 ... Q_R }
static int nd_factor_run(const NdPlan& P, NdAssembleArgs aa, double* band, double* scal, bool multi, cudaStream_t st,
                         const NdBatch& nb = NdBatch()) {
    const NdLayout lay = nd_layout(P);
    int* flags = reinterpret_cast<int*>(band + lay.flags);
    for (int s = 0; s < nb.B; ++s) {
        int* f = flags + 2 * s * nb.band;
        ASVGP_CUDA_OK(cudaMemsetAsync(f, 0, (size_t)lay.n_flag_ints * sizeof(int), st));
        ASVGP_CUDA_OK(cudaMemsetAsync(f + P.n_tiles + 1, 0x7f, sizeof(int), st));                       // first bad pivot = "none"
    }
    const int n_all = (int)P.all_tasks.size();
    aa.fronts = P.d_fronts; aa.tasks = P.d_all_tasks; aa.n_tasks = n_all; aa.idx = P.d_idx; aa.M = P.M; aa.Lpool = band;
    aa.band_stride = nb.band;
    nd_assemble_kernel<<<dim3(nd_grid_x(n_all, 148 * 16, nb.B), nb.B), 256, 0, st>>>(aa); ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    for (int lev = P.n_levels - 1; lev >= 0; --lev) {
        const int n_tasks = (int)P.factor_tasks[lev].size();
        NdFactorArgs fa{P.d_fronts, P.d_factor_tasks[lev], n_tasks, P.d_idx, P.d_pmap, band, band + lay.linv, flags, P.n_tiles,
                        nb.B, nb.band};
        if (int rc = nd_launch_persistent(nd_factor_kernel, &fa, n_tasks * nb.B, st)) return rc;
    }
    nd_scalars_kernel<<<dim3(kNdScalarBlocks, nb.B), 256, 0, st>>>(P.d_doff, P.M, band, P.d_quad_off, P.R, multi ? 2 : 1, multi ? 1 : 2,
                                                                   flags, P.n_tiles, scal, band + lay.scal, nb.band, nb.scal);
    ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

// selected inverse of every front + x_d = P^-1 b_d; returns the abort flag's address (slot 0's) for the extraction kernels
static int nd_selinv_run(const NdPlan& P, double* band, double* sig_band, double* x_out, double* work, cudaStream_t st,
                         const int** abort_flag_out, const NdBatch& nb = NdBatch()) {
    const NdLayout lay = nd_layout(P);
    int* flags = reinterpret_cast<int*>(work);
    for (int s = 0; s < nb.B; ++s)
        ASVGP_CUDA_OK(cudaMemsetAsync(flags + 2 * s * nb.work, 0, (size_t)lay.n_work_ints * sizeof(int), st));
    double* sigL = sig_band;
    double* sigU = sig_band + lay.sig_upper;
    const size_t yp_smem = (size_t)(2 * TILE_P) * sizeof(double);
    ASVGP_CUDA_OK(cudaFuncSetAttribute(nd_ypass_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)yp_smem));
    const int n_yp = (int)P.ypass_tasks.size();
    nd_ypass_kernel<<<dim3(nd_grid_x(n_yp, 148 * 3, nb.B), nb.B), kTdThreads, yp_smem, st>>>(P.d_fronts, P.d_ypass_tasks, n_yp, band,
                                                                                          band + lay.linv, sigL, nb.band, nb.sig);
    ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    for (int lev = 0; lev < P.n_levels; ++lev) {
        const int n_g = (int)P.gather_tasks[lev].size();
        NdGatherArgs ga{P.d_fronts, P.d_gather_tasks[lev], n_g, P.d_pmap, sigL, sigU, band + lay.scal, P.R, nb.band, nb.sig};
        nd_gather_kernel<<<dim3(nd_grid_x(n_g, 148 * 8, nb.B), nb.B), 256, 0, st>>>(ga); ASVGP_LAUNCHED();
        ASVGP_CUDA_OK(cudaGetLastError());
        const int n_s = (int)P.selinv_tasks[lev].size();
        if (n_s == 0) continue;
        NdSelArgs sa{P.d_fronts, P.d_selinv_tasks[lev], n_s, band, sigL, sigU, flags, P.n_tiles, P.n_cnt, nb.B, nb.band, nb.sig, nb.work};
        const int rc = nb.B > 1 ? nd_launch_persistent(nd_selinv_kernel<true>, &sa, n_s * nb.B, st)
                                : nd_launch_persistent(nd_selinv_kernel<false>, &sa, n_s, st);
        if (rc) return rc;
    }
    const int* abort_flag = flags + P.n_tiles + P.n_cnt;
    const int RM = P.M * P.R;
    nd_x_kernel<<<dim3((RM + 255) / 256, nb.B), 256, 0, st>>>(P.d_xoff, RM, sigL, band + lay.scal, abort_flag, x_out, nb.band, nb.sig,
                                                              nb.work);
    ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    *abort_flag_out = abort_flag;
    return kOk;
}

static int nd_kron_factor(const double* K1, const double* K2, const double* Gs, int m1, int m2, int order, int n_rhs, double sigma2,
                          double* band, double* rhs_io, double* scal, bool multi, void* stream) {
    const NdPlan* Pp = nullptr;
    if (int rc = nd_plan_device(m1, m2, order, n_rhs, &Pp)) return rc;
    NdAssembleArgs aa{};
    aa.K1 = K1; aa.K2 = K2; aa.Gs = Gs; aa.b = rhs_io; aa.sigma2[0] = sigma2; aa.m1 = m1; aa.m2 = m2; aa.K = order; aa.dense = nullptr;
    return nd_factor_run(*Pp, aa, band, scal, multi, static_cast<cudaStream_t>(stream));
}

static int nd_kron_selinv(double* band, int m1, int m2, int order, int n_rhs, double* sig_band, double* x_io, double* sigma_stencil,
                          double* work, void* stream) {
    const NdPlan* Pp = nullptr;
    if (int rc = nd_plan_device(m1, m2, order, n_rhs, &Pp)) return rc;
    const NdPlan& P = *Pp;
    const NdLayout lay = nd_layout(P);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int* abort_flag = nullptr;
    if (int rc = nd_selinv_run(P, band, sig_band, x_io, work, st, &abort_flag)) return rc;
    const int64_t total = (int64_t)P.M * (order + 1) * (2 * order + 1);
    nd_stencil_kernel<<<(int)std::min<int64_t>((total + 255) / 256, 148 * 16), 256, 0, st>>>(P.d_sigoff, m1, m2, order, P.R, sig_band,
                                                                                          x_io, band + lay.scal, abort_flag,
                                                                                          sigma_stencil, 0, 0, 0);
    ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

// Assembles and factorises P front by front.  band: asvgp_kron_band_doubles doubles (opaque).  rhs_io[m1 m2]: Kuf_y (read
// only here; asvgp_kron_selinv overwrites it with P^-1 Kuf_y).  scal[3] = log|P|, ||L^-1 Kuf_y||^2, info.
extern "C" int asvgp_kron_factor(const double* K1, const double* K2, const double* Gs, int m1, int m2, int order,
                                 double sigma2, double* band, double* rhs_io, double* scal, void* stream) {
    ND_CHECK_ARGS("kron_factor");
    ASVGP_REQUIRE(sigma2 > 0.0, "kron_factor: sigma2=%g", sigma2);
    return nd_kron_factor(K1, K2, Gs, m1, m2, order, 1, sigma2, band, rhs_io, scal, false, stream);
}

// From the factor (consumed: its off-diagonal tiles become Y^T): sigma_stencil[(order+1)(2 order+1) x M] = entries of P^-1
// on the stencil, x_io[M] = P^-1 Kuf_y.  sig_band: asvgp_kron_sig_doubles doubles of scratch; work: asvgp_kron_work_doubles.
// If a persistent kernel gives up waiting (abort flag), the outputs are NaN.
extern "C" int asvgp_kron_selinv(double* band, int m1, int m2, int order, double* sig_band, double* x_io,
                                 double* sigma_stencil, double* work, void* stream) {
    ND_CHECK_ARGS("kron_selinv");
    return nd_kron_selinv(band, m1, m2, order, 1, sig_band, x_io, sigma_stencil, work, stream);
}

// n_rhs right-hand sides: rhs_io[n_rhs x M] (column d at d M), scal[2 + n_rhs] = { log|P|, info, ||L^-1 b_d||^2 ... }
extern "C" int asvgp_kron_factor_multi(const double* K1, const double* K2, const double* Gs, int m1, int m2, int order, int n_rhs,
                                       double sigma2, double* band, double* rhs_io, double* scal, void* stream) {
    ND_CHECK_ARGS("kron_factor_multi");
    ND_CHECK_RHS("kron_factor_multi");
    ASVGP_REQUIRE(sigma2 > 0.0, "kron_factor_multi: sigma2=%g", sigma2);
    return nd_kron_factor(K1, K2, Gs, m1, m2, order, n_rhs, sigma2, band, rhs_io, scal, true, stream);
}

extern "C" int asvgp_kron_selinv_multi(double* band, int m1, int m2, int order, int n_rhs, double* sig_band, double* x_io,
                                       double* sigma_stencil, double* work, void* stream) {
    ND_CHECK_ARGS("kron_selinv_multi");
    ND_CHECK_RHS("kron_selinv_multi");
    return nd_kron_selinv(band, m1, m2, order, n_rhs, sig_band, x_io, sigma_stencil, work, stream);
}

// ---- B hyper-parameter settings through one plan ----------------------------------------------------------------------------------
// Every slot runs the kernels of the single-setting calls on its own buffers; the persistent launches deal the tasks of all
// slots task-major.  Slot strides are rounded to 32 doubles so that every slot's tiles keep the 256-byte alignment of the bulk
// copies.
static long long nd_slot_doubles(long long n) { return (n + 31) & ~31LL; }

static NdBatch nd_batch(const NdPlan& P, int B) {
    const NdLayout L = nd_layout(P);
    NdBatch nb;
    nb.B = B; nb.band = nd_slot_doubles(L.band_total); nb.sig = nd_slot_doubles(L.sig_total); nb.work = nd_slot_doubles(L.work_total);
    nb.scal = 2 + P.R;
    return nb;
}

#define ND_CHECK_BATCH(name) ASVGP_REQUIRE(B >= 1 && B <= ASVGP_MAX_BATCH, name ": B=%d not in 1..%d", B, ASVGP_MAX_BATCH)

extern "C" int asvgp_kron_doubles_batched(int m1, int m2, int order, int n_rhs, int B, int64_t* h_sizes) {
    ND_CHECK_ARGS("kron_doubles_batched");
    ND_CHECK_RHS("kron_doubles_batched");
    ND_CHECK_BATCH("kron_doubles_batched");
    ASVGP_REQUIRE(h_sizes != nullptr, "kron_doubles_batched: h_sizes is NULL");
    const NdPlan& P = *nd_plan_host(m1, m2, order, n_rhs);
    const NdBatch nb = nd_batch(P, B);
    h_sizes[0] = B * nb.band; h_sizes[1] = B * nb.sig; h_sizes[2] = B * nb.work;
    h_sizes[3] = (int64_t)B * n_rhs * P.M;
    h_sizes[4] = (int64_t)B * nb.scal;
    h_sizes[5] = (int64_t)B * (order + 1) * (2 * order + 1) * P.M;
    return kOk;
}

extern "C" int asvgp_kron_factor_batched(const double* K1, const double* K2, const double* Gs, const double* b, int m1, int m2,
                                         int order, int n_rhs, int B, const double* h_sigma2, double* band, int64_t band_doubles,
                                         double* scal, void* stream) {
    ND_CHECK_ARGS("kron_factor_batched");
    ND_CHECK_RHS("kron_factor_batched");
    ND_CHECK_BATCH("kron_factor_batched");
    ASVGP_REQUIRE(h_sigma2 != nullptr, "kron_factor_batched: h_sigma2 is NULL");
    ASVGP_REQUIRE(K1 != nullptr && K2 != nullptr && Gs != nullptr && b != nullptr && band != nullptr && scal != nullptr,
                  "kron_factor_batched: NULL buffer");
    for (int s = 0; s < B; ++s)
        ASVGP_REQUIRE(h_sigma2[s] > 0.0, "kron_factor_batched: slot %d: sigma2=%g must be positive", s, h_sigma2[s]);
    const NdBatch need = nd_batch(*nd_plan_host(m1, m2, order, n_rhs), B);
    ASVGP_REQUIRE(band_doubles >= B * need.band, "kron_factor_batched: band holds %lld doubles, %lld needed", (long long)band_doubles,
                  (long long)(B * need.band));
    const NdPlan* Pp = nullptr;
    if (int rc = nd_plan_device(m1, m2, order, n_rhs, &Pp)) return rc;
    NdAssembleArgs aa{};
    aa.K1 = K1; aa.K2 = K2; aa.Gs = Gs; aa.b = b; aa.m1 = m1; aa.m2 = m2; aa.K = order; aa.dense = nullptr;
    aa.k1_stride = (long long)(order + 1) * m1; aa.k2_stride = (long long)(order + 1) * m2;
    for (int s = 0; s < B; ++s) aa.sigma2[s] = h_sigma2[s];
    return nd_factor_run(*Pp, aa, band, scal, true, static_cast<cudaStream_t>(stream), need);
}

extern "C" int asvgp_kron_selinv_batched(double* band, int m1, int m2, int order, int n_rhs, int B, int64_t band_doubles,
                                         double* sig_band, int64_t sig_doubles, double* work, int64_t work_doubles, double* x_out,
                                         double* sigma_stencil, void* stream) {
    ND_CHECK_ARGS("kron_selinv_batched");
    ND_CHECK_RHS("kron_selinv_batched");
    ND_CHECK_BATCH("kron_selinv_batched");
    ASVGP_REQUIRE(band != nullptr && sig_band != nullptr && work != nullptr && x_out != nullptr && sigma_stencil != nullptr,
                  "kron_selinv_batched: NULL buffer");
    const NdBatch nb = nd_batch(*nd_plan_host(m1, m2, order, n_rhs), B);
    ASVGP_REQUIRE(band_doubles >= B * nb.band && sig_doubles >= B * nb.sig && work_doubles >= B * nb.work,
                  "kron_selinv_batched: buffers of %lld / %lld / %lld doubles, %lld / %lld / %lld needed", (long long)band_doubles,
                  (long long)sig_doubles, (long long)work_doubles, (long long)(B * nb.band), (long long)(B * nb.sig),
                  (long long)(B * nb.work));
    const NdPlan* Pp = nullptr;
    if (int rc = nd_plan_device(m1, m2, order, n_rhs, &Pp)) return rc;
    const NdPlan& P = *Pp;
    const NdLayout lay = nd_layout(P);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int* abort_flag = nullptr;
    if (int rc = nd_selinv_run(P, band, sig_band, x_out, work, st, &abort_flag, nb)) return rc;
    const int64_t total = (int64_t)P.M * (order + 1) * (2 * order + 1);
    nd_stencil_kernel<<<dim3(nd_grid_x((total + 255) / 256, 148 * 16, B), B), 256, 0, st>>>(P.d_sigoff, m1, m2, order, P.R, sig_band, x_out,
                                                                                         band + lay.scal, abort_flag, sigma_stencil,
                                                                                         nb.band, nb.sig, nb.work);
    ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

// ---- dense symmetric positive definite matrices on the same kernels (one front) -----------------------------------------------------
// What GPR_additive needs (reference gpr.py:192-195, 221-231: tf.linalg.cholesky / triangular_solve of a DENSE (sum m_d)^2
// matrix): log|A|, b^T A^-1 b, A^-1 b and A^-1, from the tile-DAG factorisation and the blocked Takahashi recursion above.
extern "C" int64_t asvgp_dense_band_doubles(int n) {
    if (n <= 0 || n > 32768) return -1;
    return nd_layout(*nd_plan_host(n, 1, -1)).band_total;
}
extern "C" int64_t asvgp_dense_sig_doubles(int n) {
    if (n <= 0 || n > 32768) return -1;
    return nd_layout(*nd_plan_host(n, 1, -1)).sig_total;
}
extern "C" int64_t asvgp_dense_work_doubles(int n) {
    if (n <= 0 || n > 32768) return -1;
    return nd_layout(*nd_plan_host(n, 1, -1)).work_total;
}

#define ND_CHECK_DENSE(name) ASVGP_REQUIRE(n > 0 && n <= 32768, name ": n=%d", n)

extern "C" int asvgp_dense_doubles_multi(int n, int n_rhs, int64_t* h_sizes) {
    ND_CHECK_DENSE("dense_doubles_multi");
    ND_CHECK_RHS("dense_doubles_multi");
    nd_sizes(*nd_plan_host(n, 1, -1, n_rhs), h_sizes);
    return kOk;
}

static int nd_dense_factor(const double* A, int n, int n_rhs, const double* rhs, double* band, double* scal, bool multi, void* stream) {
    const NdPlan* Pp = nullptr;
    if (int rc = nd_plan_device(n, 1, -1, n_rhs, &Pp)) return rc;
    NdAssembleArgs aa{};
    aa.b = rhs; aa.sigma2[0] = 1.0; aa.m1 = n; aa.m2 = 1; aa.K = 0; aa.dense = A;
    return nd_factor_run(*Pp, aa, band, scal, multi, static_cast<cudaStream_t>(stream));
}

// A: n x n row-major (lower triangle read), rhs[n].  scal[3] = log|A|, rhs^T A^-1 rhs, info (0 ok, j+1 = row of the first
// non-positive pivot, -1 internal time-out).
extern "C" int asvgp_dense_factor(const double* A, int n, const double* rhs, double* band, double* scal, void* stream) {
    ND_CHECK_DENSE("dense_factor");
    return nd_dense_factor(A, n, 1, rhs, band, scal, false, stream);
}

// rhs[n_rhs x n] (column d at d n); scal[2 + n_rhs] = { log|A|, info, rhs_d^T A^-1 rhs_d ... }
extern "C" int asvgp_dense_factor_multi(const double* A, int n, int n_rhs, const double* rhs, double* band, double* scal,
                                        void* stream) {
    ND_CHECK_DENSE("dense_factor_multi");
    ND_CHECK_RHS("dense_factor_multi");
    return nd_dense_factor(A, n, n_rhs, rhs, band, scal, true, stream);
}

namespace asvgp {
// inv[i * n + j] = Sigma'(i, j) - tau sum_d x_d,i x_d,j for the single front of a dense plan (diagonal tiles averaged with their
// mirror)
__global__ void __launch_bounds__(256) nd_dense_extract_kernel(FrontDesc f, int n, int R, const double* __restrict__ sig_lower,
                                                               const double* __restrict__ x, const double* __restrict__ scal_keep,
                                                               const int* __restrict__ abort_flag, double* __restrict__ inv) {
    const double tau = scal_keep[1];
    const bool aborted = *abort_flag != 0;
    const long long total = (long long)n * n;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(t / n), j = (int)(t % n);
        const int hi = max(i, j), lo = min(i, j);
        const double* tile = sig_lower + front_tile(f, hi / NB, lo / NB) * TILE_P;
        double v = __ldcg(tile + (lo % NB) * LDT + hi % NB);
        if (hi / NB == lo / NB) v = 0.5 * (v + __ldcg(tile + (hi % NB) * LDT + lo % NB));
        if (R == 1) inv[t] = aborted ? nan("") : v - tau * x[i] * x[j];       // the single-rhs expression as it was
        else inv[t] = aborted ? nan("") : v - nd_rank_correction(x, n, R, tau, i, j);
    }
}
}  // namespace asvgp

static int nd_dense_selinv(double* band, int n, int n_rhs, double* sig_band, double* x_out, double* inv_out, double* work,
                           void* stream) {
    const NdPlan* Pp = nullptr;
    if (int rc = nd_plan_device(n, 1, -1, n_rhs, &Pp)) return rc;
    const NdPlan& P = *Pp;
    const NdLayout lay = nd_layout(P);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int* abort_flag = nullptr;
    if (int rc = nd_selinv_run(P, band, sig_band, x_out, work, st, &abort_flag)) return rc;
    const int64_t total = (int64_t)n * n;
    nd_dense_extract_kernel<<<(int)std::min<int64_t>((total + 255) / 256, 148 * 16), 256, 0, st>>>(P.fronts[0], n, P.R, sig_band, x_out,
                                                                                                 band + lay.scal, abort_flag, inv_out);
    ASVGP_LAUNCHED();
    ASVGP_CUDA_OK(cudaGetLastError());
    return kOk;
}

// band is CONSUMED.  x_out[n] = A^-1 rhs, inv_out[n x n] = A^-1 (full symmetric, row-major).
extern "C" int asvgp_dense_selinv(double* band, int n, double* sig_band, double* x_out, double* inv_out, double* work, void* stream) {
    ND_CHECK_DENSE("dense_selinv");
    return nd_dense_selinv(band, n, 1, sig_band, x_out, inv_out, work, stream);
}

// x_out[n_rhs x n]: x_out[d n + i] = (A^-1 rhs_d)_i
extern "C" int asvgp_dense_selinv_multi(double* band, int n, int n_rhs, double* sig_band, double* x_out, double* inv_out,
                                        double* work, void* stream) {
    ND_CHECK_DENSE("dense_selinv_multi");
    ND_CHECK_RHS("dense_selinv_multi");
    return nd_dense_selinv(band, n, n_rhs, sig_band, x_out, inv_out, work, stream);
}
