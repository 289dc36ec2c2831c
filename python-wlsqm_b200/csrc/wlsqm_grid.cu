// wlsqm_grid.cu -- uniform-grid spatial search on the device: k nearest neighbours of every point of a cloud
// (neighbourhood construction) and of arbitrary query points (nearest local model).
//
// This is the step *before* the fitting path in the reference's pipeline, done there on the host with
// scipy.spatial.cKDTree (examples/expertsolver_example.py:51-66: hoods = tree.query(x, k+1)[1][:,1:];
// wlsqm/fitter/expert.pyx:676-681,837: tree.query(x, k=1)).  Results are the exact k nearest neighbours,
// ordered by (distance, index); they coincide with cKDTree's wherever distances are distinct (ties are
// ordered arbitrarily by cKDTree -- tests/test_gpu_grid.py compares index for index on random clouds).
//
// Build: bounding box -> cell size for ~2 points per cell -> cell id per point -> stable radix sort of
// (cell, index) pairs (cub) -> per-cell start offsets (histogram + exclusive scan) -> coordinates gathered
// into sorted order.  Query: one thread per query walks the cell shells around its own cell, keeps the k best
// candidates in a sorted list, and stops when the k-th distance is below the distance to the unvisited region.
// Ball search (cKDTree.query_ball_point, examples/wlsqm_example.py:100-132): one thread per query walks the cell box
// of its ball twice -- count, then fill CSR rows -- and cub's segmented sort orders the rows; max_k runs the k-nearest
// walk bounded by r.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <new>
#include <string>

#include <cub/cub.cuh>

#include "../../include/wlsqm_b200.h"
#include "wlsqm_grid.h"
#include "wlsqm_kernels.h"
#include "wlsqm_mem.h"

using namespace wlsqm;

struct wlsqm_grid {
    int dim = 0, device = 0;
    long long n = 0, ncells = 0;
    GridView v{};
    int* cell_start = nullptr;
    int* sorted_idx = nullptr;
    double* sorted_x = nullptr;
    cudaStream_t stream = nullptr;
    long long bytes = 0;
};

namespace wlsqm {
GridView grid_view(const wlsqm_grid* g) { return g->v; }
int grid_device(const wlsqm_grid* g) { return g->device; }
}  // namespace wlsqm

namespace {

int gfail(int code, const char* msg) {
    wlsqm::set_last_error(msg);
    return code;
}

#define GCU(expr)                                                                                   \
    do {                                                                                            \
        cudaError_t e__ = (expr);                                                                   \
        if (e__ != cudaSuccess) {                                                                   \
            std::string m__ = std::string(#expr) + ": " + cudaGetErrorString(e__);                  \
            return gfail(e__ == cudaErrorMemoryAllocation ? WLSQM_E_MEMORY : WLSQM_E_CUDA, m__.c_str()); \
        }                                                                                           \
    } while (0)

// order-preserving map double -> uint64 (for atomicMin / atomicMax)
__device__ __forceinline__ unsigned long long enc(double x) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(x);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ULL);
}
inline double dec(unsigned long long u) {
    const unsigned long long b = (u >> 63) ? (u & 0x7fffffffffffffffULL) : ~u;
    double x;
    memcpy(&x, &b, 8);
    return x;
}

__global__ void bbox_kernel(const double* __restrict__ x, long long s0, long long n, int dim, unsigned long long* mm) {
    double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        for (int d = 0; d < dim; ++d) {
            const double v = x[i * s0 + d];
            if (fabs(v) <= 1.79769313486231570e308) {     // NaN and +/-inf coordinates do not shape the box
                lo[d] = fmin(lo[d], v);
                hi[d] = fmax(hi[d], v);
            }
        }
    for (int d = 0; d < dim; ++d) {
        for (int o = 16; o > 0; o >>= 1) {
            lo[d] = fmin(lo[d], __shfl_xor_sync(0xffffffffu, lo[d], o));
            hi[d] = fmax(hi[d], __shfl_xor_sync(0xffffffffu, hi[d], o));
        }
        if ((threadIdx.x & 31) == 0) {
            atomicMin(&mm[d], enc(lo[d]));
            atomicMax(&mm[3 + d], enc(hi[d]));
        }
    }
}

__global__ void cell_id_kernel(GridView g, const double* __restrict__ x, long long s0, int* __restrict__ cid,
                               int* __restrict__ idx, int* __restrict__ counts) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= g.n) return;
    int c = 0;
    for (int d = g.dim - 1; d >= 0; --d) c = c * g.dims[d] + grid_cell_coord(g, d, x[i * s0 + d]);
    cid[i] = c;
    idx[i] = (int)i;
    atomicAdd(&counts[c], 1);
}

__global__ void gather_sorted_kernel(long long n, int dim, const double* __restrict__ x, long long s0,
                                     const int* __restrict__ sorted_idx, double* __restrict__ xs) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * dim) return;
    const long long p = t / dim;
    const int d = (int)(t - p * dim);
    xs[t] = x[(long long)sorted_idx[p] * s0 + d];
}

// ---- ball search: the membership rule of include/wlsqm_b200.h ------------------------------------------------
// d2 is summed over the axes in axis order with every difference, square and sum rounded on its own (no contraction
// into FMAs), so that the count and fill passes, the capped walk and a numpy restatement all agree bit for bit.
template <int DIM>
__device__ __forceinline__ double ball_d2(const GridView& g, long long p, const double (&q)[DIM]) {
    double d2 = 0.0;
#pragma unroll
    for (int d = 0; d < DIM; ++d) {
        const double dd = __dsub_rn(g.sorted_x[p * DIM + d], q[d]);
        d2 = __dadd_rn(d2, __dmul_rn(dd, dd));
    }
    return d2;
}

// grid point p (at d2 from a finite query) is a member: d2 <= r2, and a point with a non-finite coordinate never is
// (it can only pass d2 <= r2 when r2 is infinite: NaN fails the comparison, +/-inf gives d2 = inf)
template <int DIM>
__device__ __forceinline__ bool ball_member(const GridView& g, long long p, double d2, double r2) {
    if (!(d2 <= r2)) return false;
    if (d2 < INFINITY) return true;
    bool finite = true;
#pragma unroll
    for (int d = 0; d < DIM; ++d) finite = finite && fabs(g.sorted_x[p * DIM + d]) <= 1.79769313486231570e308;
    return finite;
}

struct BallArgs {
    const double* xq;       // NULL: the grid's own points
    long long xq_s0, nq;
    const double* r;        // [nq] with stride r_s0 (0: one radius); indexed by point index for the grid's own points
    long long r_s0;
    int exclude_self;
    int* bad;               // set when a radius is negative or NaN
};

// Query t of a launch: its output row qi, coordinates, squared radius and the half-width w of a box that holds every
// member.  A member has fl(dd^2) <= fl(r^2) on every axis, so |dd| <= r (1 + 2^-52) when r^2 is normal and
// |dd| < sqrt(DBL_MIN) < 1.5e-154 when it is not; w adds a relative 2^-40 to that bound.  false: the row is empty
// (a non-finite query coordinate, or an invalid radius, which is flagged).
template <int DIM, bool SELF>
__device__ __forceinline__ bool ball_query(const GridView& g, const BallArgs& a, long long t, long long& qi,
                                           double (&q)[DIM], double& r2, double& w) {
    if (SELF) {
        qi = g.sorted_idx[t];
#pragma unroll
        for (int d = 0; d < DIM; ++d) q[d] = g.sorted_x[t * DIM + d];
    } else {
        qi = t;
#pragma unroll
        for (int d = 0; d < DIM; ++d) q[d] = a.xq[t * a.xq_s0 + d];
    }
    const double r = a.r[qi * a.r_s0];
    if (!(r >= 0.0)) {
        atomicExch(a.bad, 1);
        return false;
    }
    r2 = __dmul_rn(r, r);
    w = fmax(r, 1.5e-154) * (1.0 + 0x1p-40);
    bool finite = true;
#pragma unroll
    for (int d = 0; d < DIM; ++d) finite = finite && fabs(q[d]) <= 1.79769313486231570e308;
    return finite;
}

// The cells that hold every member: [cell(q - w'), cell(q + w')] per axis with w' = w + 2^-40 |q|, which covers the
// rounding of q -/+ w.  Cell coordinates are monotone in x (the same grid_cell_coord that placed the points), so a
// member can only lie outside the box of the exact half-width if rounding cuts it, and the slack moves the bound by a
// cell exactly where it does (members on cell edges and at exactly r).  The box is exact in cell coordinates: it does
// not depend on where the cell edges fall in floating point.
template <int DIM>
__device__ __forceinline__ void ball_box(const GridView& g, const double (&q)[DIM], double w, int (&c0)[3], int (&c1)[3]) {
#pragma unroll
    for (int d = 0; d < DIM; ++d) {
        const double s = w + 0x1p-40 * fabs(q[d]);
        c0[d] = grid_cell_coord(g, d, q[d] - s);
        c1[d] = grid_cell_coord(g, d, q[d] + s);
    }
}

// Every member of the ball, in cell order: visit(p, d2) for its sorted position p, over the cells of ball_box.
// self_pos: the sorted position excluded (exclude_self), or -1.  The cells of one x-row are one contiguous range of
// sorted positions.
template <int DIM, class F>
__device__ __forceinline__ void ball_walk(const GridView& g, const double (&q)[DIM], double r2, double w, int self_pos,
                                          F&& visit) {
    int c0[3] = {0, 0, 0}, c1[3] = {0, 0, 0};
    ball_box<DIM>(g, q, w, c0, c1);
    for (int cz = c0[2]; cz <= c1[2]; ++cz)
        for (int cy = c0[1]; cy <= c1[1]; ++cy) {
            const long long row = ((long long)cz * g.dims[1] + cy) * g.dims[0];
            const int p1 = g.cell_start[row + c1[0] + 1];
            for (int p = g.cell_start[row + c0[0]]; p < p1; ++p) {
                const double d2 = ball_d2<DIM>(g, p, q);
                if (p != self_pos && ball_member<DIM>(g, p, d2, r2)) visit(p, d2);
            }
        }
}

// Uncapped ball search, pass 1: the number of members of every row.  SELF: the queries are the grid's own points,
// visited in sorted (cell) order as in knn_kernel.
template <int DIM, bool SELF>
__global__ void __launch_bounds__(128) ball_count_kernel(GridView g, BallArgs a, long long* __restrict__ count64,
                                                         int32_t* __restrict__ count32) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.nq) return;
    long long qi;
    double q[DIM], r2, w;
    long long c = 0;
    if (ball_query<DIM, SELF>(g, a, t, qi, q, r2, w))
        ball_walk<DIM>(g, q, r2, w, (SELF && a.exclude_self) ? (int)t : -1, [&](int, double) { ++c; });
    count64[qi] = c;
    if (count32) count32[qi] = (int32_t)c;
}

// Pass 2: the same walk writes the members' indices (and d2, for the distance order) into row qi in cell order,
// never past rowptr[qi + 1].
template <int DIM, bool SELF>
__global__ void __launch_bounds__(128) ball_fill_kernel(GridView g, BallArgs a, const int64_t* __restrict__ rowptr,
                                                        int32_t* __restrict__ col, double* __restrict__ col_d2) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.nq) return;
    long long qi;
    double q[DIM], r2, w;
    if (!ball_query<DIM, SELF>(g, a, t, qi, q, r2, w)) return;
    const long long pos = rowptr[qi];
    int32_t* out = col + pos;
    int32_t* const out_end = col + rowptr[qi + 1];
    double* out_d2 = col_d2 ? col_d2 + pos : nullptr;
    ball_walk<DIM>(g, q, r2, w, (SELF && a.exclude_self) ? (int)t : -1, [&](int p, double d2) {
        if (out < out_end) {
            *out++ = g.sorted_idx[p];
            if (out_d2) *out_d2++ = d2;
        }
    });
}

// k nearest grid points of every query.  SELF: the queries are the grid's own points, visited in sorted (cell)
// order so that the threads of a warp walk the same cells; the point itself is skipped when exclude_self.
template <int DIM, int KMAX, bool SELF>
__global__ void __launch_bounds__(128) knn_kernel(GridView g, const double* __restrict__ xq, long long xq_s0, long long nq,
                                                  int k, int exclude_self, int32_t* __restrict__ out32,
                                                  int64_t* __restrict__ out64, double* __restrict__ out_d2) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nq) return;
    double q[DIM];
    long long qi;      // row of the output
    if (SELF) {
        qi = g.sorted_idx[t];
#pragma unroll
        for (int d = 0; d < DIM; ++d) q[d] = g.sorted_x[t * DIM + d];
    } else {
        qi = t;
#pragma unroll
        for (int d = 0; d < DIM; ++d) q[d] = xq[t * xq_s0 + d];
    }
    int cq[DIM];
#pragma unroll
    for (int d = 0; d < DIM; ++d) cq[d] = grid_cell_coord(g, d, q[d]);

    double bd[KMAX];
    int bi[KMAX];
    int cnt = 0;
    double worst = INFINITY;
    int worst_i = 0x7fffffff;
    const int self = (SELF && exclude_self) ? (int)qi : -1;
    int maxr = 0;
#pragma unroll
    for (int d = 0; d < DIM; ++d) maxr = max(maxr, max(cq[d], g.dims[d] - 1 - cq[d]));

    for (int r = 0; r <= maxr; ++r) {
        // cells whose Chebyshev distance from the query's cell is exactly r
        const int z0 = DIM >= 3 ? max(cq[DIM >= 3 ? 2 : 0] - r, 0) : 0;
        const int z1 = DIM >= 3 ? min(cq[DIM >= 3 ? 2 : 0] + r, g.dims[2] - 1) : 0;
        const int y0 = DIM >= 2 ? max(cq[DIM >= 2 ? 1 : 0] - r, 0) : 0;
        const int y1 = DIM >= 2 ? min(cq[DIM >= 2 ? 1 : 0] + r, g.dims[1] - 1) : 0;
        const int x0 = max(cq[0] - r, 0), x1 = min(cq[0] + r, g.dims[0] - 1);
        for (int cz = z0; cz <= z1; ++cz) {
            const bool fz = DIM >= 3 && abs(cz - cq[DIM >= 3 ? 2 : 0]) == r;
            for (int cy = y0; cy <= y1; ++cy) {
                const bool fy = fz || (DIM >= 2 && abs(cy - cq[DIM >= 2 ? 1 : 0]) == r);
                // on a face of the shell the whole x range belongs to it, otherwise only its two end cells
                const int step = fy ? 1 : max(x1 - x0, 1);
                for (int cx = x0; cx <= x1; cx += step) {
                    if (!fy && abs(cx - cq[0]) != r) continue;
                    const long long cell = ((long long)cz * g.dims[1] + cy) * g.dims[0] + cx;
                    const int p1 = g.cell_start[cell + 1];
                    for (int p = g.cell_start[cell]; p < p1; ++p) {
                        double d2 = 0.0;
#pragma unroll
                        for (int d = 0; d < DIM; ++d) {
                            const double dd = g.sorted_x[(long long)p * DIM + d] - q[d];
                            d2 += dd * dd;
                        }
                        const int id = g.sorted_idx[p];
                        if (id == self || !(d2 < INFINITY)) continue;     // (points with NaN / inf coordinates are nobody's neighbour)
                        if (cnt == k && !(d2 < worst || (d2 == worst && id < worst_i))) continue;
                        int j = cnt < k ? cnt : k - 1;
                        while (j > 0 && (bd[j - 1] > d2 || (bd[j - 1] == d2 && bi[j - 1] > id))) {
                            bd[j] = bd[j - 1];
                            bi[j] = bi[j - 1];
                            --j;
                        }
                        bd[j] = d2;
                        bi[j] = id;
                        if (cnt < k) ++cnt;
                        if (cnt == k) { worst = bd[k - 1]; worst_i = bi[k - 1]; }
                    }
                }
            }
        }
        if (cnt == k) {
            // every unvisited point lies outside the block of visited cells: at least `margin` away
            double margin = INFINITY;
#pragma unroll
            for (int d = 0; d < DIM; ++d) {
                if (cq[d] - r > 0) margin = fmin(margin, q[d] - (g.lo[d] + (double)(cq[d] - r) * g.h));
                if (cq[d] + r < g.dims[d] - 1) margin = fmin(margin, (g.lo[d] + (double)(cq[d] + r + 1) * g.h) - q[d]);
            }
            // (the cell edges carry rounding of order ulp(extent): keep one more shell unless clearly inside)
            if (margin > 0.0 && worst < margin * margin * (1.0 - 1e-12)) break;
        }
    }
    for (int j = 0; j < k; ++j) {
        const int id = j < cnt ? bi[j] : (int)g.n;          // missing neighbours are reported as n (like cKDTree)
        if (out32) out32[qi * k + j] = id;
        if (out64) out64[qi * k + j] = id;
        if (out_d2) out_d2[qi * k + j] = j < cnt ? bd[j] : INFINITY;
    }
}

template <int DIM, bool SELF>
cudaError_t launch_knn_k(const GridView& g, const double* xq, long long s0, long long nq, int k, int excl, int32_t* o32,
                         int64_t* o64, double* od2, cudaStream_t st) {
    const int threads = 128;
    const unsigned blocks = (unsigned)((nq + threads - 1) / threads);
    if (k <= 8) knn_kernel<DIM, 8, SELF><<<blocks, threads, 0, st>>>(g, xq, s0, nq, k, excl, o32, o64, od2);
    else if (k <= 32) knn_kernel<DIM, 32, SELF><<<blocks, threads, 0, st>>>(g, xq, s0, nq, k, excl, o32, o64, od2);
    else if (k <= 64) knn_kernel<DIM, 64, SELF><<<blocks, threads, 0, st>>>(g, xq, s0, nq, k, excl, o32, o64, od2);
    else knn_kernel<DIM, 128, SELF><<<blocks, threads, 0, st>>>(g, xq, s0, nq, k, excl, o32, o64, od2);
    return cudaGetLastError();
}

template <int DIM>
cudaError_t launch_knn_d(const GridView& g, const double* xq, long long s0, long long nq, int k, int excl, int32_t* o32,
                         int64_t* o64, double* od2, cudaStream_t st) {
    if (xq) return launch_knn_k<DIM, false>(g, xq, s0, nq, k, excl, o32, o64, od2, st);
    return launch_knn_k<DIM, true>(g, nullptr, 0, nq, k, excl, o32, o64, od2, st);
}

// Capped ball search (max_k = k): knn_kernel's shell walk bounded by r.  Only members of the ball (ball_member, with d2
// as ball_d2) are candidates.  The shells end where they cover ball_box, the same cells the uncapped walk reads, so
// no member is missed however far the cloud lies from the origin.  The early stop once the k-th distance is below the
// unvisited region allows for the rounding of the cell edges lo + c h: it subtracts 2^-40 (|q| + |lo| + |edge|) from
// the margin (knn_kernel's relative 1e-12 alone does not cover clouds far from the origin).  rowptr == NULL: the count pass (count64 / count32 as in ball_count_kernel); otherwise row qi is
// written in (d2, index) order, never past rowptr[qi + 1].  (A separate kernel: sharing the walk with knn_kernel
// through templates or a device function changed knn_kernel's register allocation.)
template <int DIM, int KMAX, bool SELF>
__global__ void __launch_bounds__(128) ball_knn_kernel(GridView g, BallArgs a, int k, long long* __restrict__ count64,
                                                       int32_t* __restrict__ count32, const int64_t* __restrict__ rowptr,
                                                       int32_t* __restrict__ col) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.nq) return;
    double q[DIM], r2, w;
    long long qi;      // row of the output
    if (!ball_query<DIM, SELF>(g, a, t, qi, q, r2, w)) {
        if (!rowptr) {
            count64[qi] = 0;
            if (count32) count32[qi] = 0;
        }
        return;
    }
    int cq[DIM];
    int maxr = 0;     // the shell that completes ball_box
    {
        int c0[3] = {0, 0, 0}, c1[3] = {0, 0, 0};
        ball_box<DIM>(g, q, w, c0, c1);
#pragma unroll
        for (int d = 0; d < DIM; ++d) {
            cq[d] = grid_cell_coord(g, d, q[d]);
            maxr = max(maxr, max(cq[d] - c0[d], c1[d] - cq[d]));
        }
    }

    double bd[KMAX];
    int bi[KMAX];
    int cnt = 0;
    double worst = INFINITY;
    int worst_i = 0x7fffffff;
    const int self = (SELF && a.exclude_self) ? (int)qi : -1;

    for (int r = 0; r <= maxr; ++r) {
        // cells whose Chebyshev distance from the query's cell is exactly r
        const int z0 = DIM >= 3 ? max(cq[DIM >= 3 ? 2 : 0] - r, 0) : 0;
        const int z1 = DIM >= 3 ? min(cq[DIM >= 3 ? 2 : 0] + r, g.dims[2] - 1) : 0;
        const int y0 = DIM >= 2 ? max(cq[DIM >= 2 ? 1 : 0] - r, 0) : 0;
        const int y1 = DIM >= 2 ? min(cq[DIM >= 2 ? 1 : 0] + r, g.dims[1] - 1) : 0;
        const int x0 = max(cq[0] - r, 0), x1 = min(cq[0] + r, g.dims[0] - 1);
        for (int cz = z0; cz <= z1; ++cz) {
            const bool fz = DIM >= 3 && abs(cz - cq[DIM >= 3 ? 2 : 0]) == r;
            for (int cy = y0; cy <= y1; ++cy) {
                const bool fy = fz || (DIM >= 2 && abs(cy - cq[DIM >= 2 ? 1 : 0]) == r);
                // on a face of the shell the whole x range belongs to it, otherwise only its two end cells
                const int step = fy ? 1 : max(x1 - x0, 1);
                for (int cx = x0; cx <= x1; cx += step) {
                    if (!fy && abs(cx - cq[0]) != r) continue;
                    const long long cell = ((long long)cz * g.dims[1] + cy) * g.dims[0] + cx;
                    const int p1 = g.cell_start[cell + 1];
                    for (int p = g.cell_start[cell]; p < p1; ++p) {
                        const double d2 = ball_d2<DIM>(g, p, q);
                        if (!ball_member<DIM>(g, p, d2, r2)) continue;
                        const int id = g.sorted_idx[p];
                        if (id == self) continue;
                        if (cnt == k && !(d2 < worst || (d2 == worst && id < worst_i))) continue;
                        int j = cnt < k ? cnt : k - 1;
                        while (j > 0 && (bd[j - 1] > d2 || (bd[j - 1] == d2 && bi[j - 1] > id))) {
                            bd[j] = bd[j - 1];
                            bi[j] = bi[j - 1];
                            --j;
                        }
                        bd[j] = d2;
                        bi[j] = id;
                        if (cnt < k) ++cnt;
                        if (cnt == k) { worst = bd[k - 1]; worst_i = bi[k - 1]; }
                    }
                }
            }
        }
        if (cnt == k && r < maxr) {
            // every unvisited point lies outside the block of visited cells: at least `margin` away, less the rounding
            // of the cell edges and of the differences
            double margin = INFINITY;
#pragma unroll
            for (int d = 0; d < DIM; ++d) {
                const double slack = 0x1p-40 * (fabs(q[d]) + fabs(g.lo[d]));
                if (cq[d] - r > 0) {
                    const double e = g.lo[d] + (double)(cq[d] - r) * g.h;
                    margin = fmin(margin, (q[d] - e) - (slack + 0x1p-40 * fabs(e)));
                }
                if (cq[d] + r < g.dims[d] - 1) {
                    const double e = g.lo[d] + (double)(cq[d] + r + 1) * g.h;
                    margin = fmin(margin, (e - q[d]) - (slack + 0x1p-40 * fabs(e)));
                }
            }
            if (margin > 0.0 && worst < margin * margin * (1.0 - 1e-12)) break;
        }
    }
    if (!rowptr) {
        count64[qi] = cnt;
        if (count32) count32[qi] = cnt;
        return;
    }
    const long long pos = rowptr[qi], end = rowptr[qi + 1];
    for (int j = 0; j < cnt && pos + j < end; ++j) col[pos + j] = bi[j];
}

// rowptr == NULL: the count pass; otherwise the fill pass (col_d2: d2 beside col, uncapped only)
template <int DIM, bool SELF>
cudaError_t launch_ball_s(const GridView& g, const BallArgs& a, int max_k, long long* c64, int32_t* c32,
                          const int64_t* rowptr, int32_t* col, double* col_d2, cudaStream_t st) {
    const unsigned blocks = (unsigned)((a.nq + 127) / 128);
    if (max_k == 0) {
        if (!rowptr) ball_count_kernel<DIM, SELF><<<blocks, 128, 0, st>>>(g, a, c64, c32);
        else ball_fill_kernel<DIM, SELF><<<blocks, 128, 0, st>>>(g, a, rowptr, col, col_d2);
    } else if (max_k <= 8) ball_knn_kernel<DIM, 8, SELF><<<blocks, 128, 0, st>>>(g, a, max_k, c64, c32, rowptr, col);
    else if (max_k <= 32) ball_knn_kernel<DIM, 32, SELF><<<blocks, 128, 0, st>>>(g, a, max_k, c64, c32, rowptr, col);
    else if (max_k <= 64) ball_knn_kernel<DIM, 64, SELF><<<blocks, 128, 0, st>>>(g, a, max_k, c64, c32, rowptr, col);
    else ball_knn_kernel<DIM, 128, SELF><<<blocks, 128, 0, st>>>(g, a, max_k, c64, c32, rowptr, col);
    return cudaGetLastError();
}

cudaError_t launch_ball(const GridView& g, const BallArgs& a, int max_k, long long* c64, int32_t* c32,
                        const int64_t* rowptr, int32_t* col, double* col_d2, cudaStream_t st) {
    if (a.nq == 0) return cudaSuccess;
    switch (g.dim * 2 + (a.xq ? 0 : 1)) {
        case 2: return launch_ball_s<1, false>(g, a, max_k, c64, c32, rowptr, col, col_d2, st);
        case 3: return launch_ball_s<1, true>(g, a, max_k, c64, c32, rowptr, col, col_d2, st);
        case 4: return launch_ball_s<2, false>(g, a, max_k, c64, c32, rowptr, col, col_d2, st);
        case 5: return launch_ball_s<2, true>(g, a, max_k, c64, c32, rowptr, col, col_d2, st);
        case 6: return launch_ball_s<3, false>(g, a, max_k, c64, c32, rowptr, col, col_d2, st);
        default: return launch_ball_s<3, true>(g, a, max_k, c64, c32, rowptr, col, col_d2, st);
    }
}

int is_dev(const void* p) {
    if (!p) return 0;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

}  // namespace

extern "C" {

int wlsqm_grid_destroy(wlsqm_grid_t* g) {
    if (!g) return WLSQM_OK;
    cudaSetDevice(g->device);
    if (g->stream) cudaStreamSynchronize(g->stream);
    dev_free(g->cell_start); dev_free(g->sorted_idx); dev_free(g->sorted_x);
    if (g->stream) cudaStreamDestroy(g->stream);
    cudaGetLastError();
    delete g;
    return WLSQM_OK;
}

int wlsqm_grid_create(int dimension, int64_t n, const double* x, int64_t x_s0, int device, wlsqm_grid_t** out) {
    if (!out) return gfail(WLSQM_E_VALUE, "out is NULL");
    *out = nullptr;
    if (dimension < 1 || dimension > 3) return gfail(WLSQM_E_VALUE, "dimension must be 1, 2 or 3");
    if (n < 1 || n > 2000000000LL) return gfail(WLSQM_E_VALUE, "the grid needs between 1 and 2e9 points");
    if (!x) return gfail(WLSQM_E_VALUE, "x is NULL");
    if (wlsqm_device_count() < 1) return gfail(WLSQM_E_CUDA, "no CUDA device available (there is no CPU fallback)");
    GCU(cudaSetDevice(device));
    wlsqm_grid* g = new (std::nothrow) wlsqm_grid();
    if (!g) return gfail(WLSQM_E_MEMORY, "out of host memory");
    g->dim = dimension; g->device = device; g->n = n;
    cudaError_t e = cudaStreamCreateWithFlags(&g->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { delete g; return gfail(WLSQM_E_CUDA, cudaGetErrorString(e)); }
    cudaStream_t st = g->stream;
    auto bail = [&](int rc) { wlsqm_grid_destroy(g); return rc; };
    // the points may still be being produced on the caller's stream (device arrays)
    if (order_after_caller(st) != cudaSuccess) { cudaGetLastError(); cudaStreamSynchronize(caller_stream()); }

    // the points on the device (a host array is staged; only the sorted copy is kept)
    double* xd = nullptr;
    const double* xdev = x;
    long long s0 = x_s0;
    if (!is_dev(x)) {
        if (dev_alloc((void**)&xd, (size_t)n * dimension * 8) != cudaSuccess) return bail(gfail(WLSQM_E_MEMORY, "cudaMalloc failed (grid points)"));
        e = cudaMemcpy2DAsync(xd, (size_t)dimension * 8, x, (size_t)x_s0 * 8, (size_t)dimension * 8, (size_t)n, cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) { dev_free(xd); return bail(gfail(WLSQM_E_CUDA, cudaGetErrorString(e))); }
        xdev = xd;
        s0 = dimension;
    }
    unsigned long long* mm = nullptr;
    int *cid = nullptr, *idx = nullptr, *cid_s = nullptr, *counts = nullptr;
    void* tmp = nullptr;
    auto cleanup = [&]() { dev_free(xd); dev_free(mm); dev_free(cid); dev_free(idx); dev_free(cid_s); dev_free(counts); dev_free(tmp); };
    auto fail_here = [&](int code, const char* msg) { cudaStreamSynchronize(st); cleanup(); return bail(gfail(code, msg)); };

    // ---- bounding box -> cell size ----------------------------------------------------------------------
    if (dev_alloc((void**)&mm, 6 * 8) != cudaSuccess) return fail_here(WLSQM_E_MEMORY, "cudaMalloc failed");
    unsigned long long init[6] = {~0ULL, ~0ULL, ~0ULL, 0ULL, 0ULL, 0ULL};
    cudaMemcpyAsync(mm, init, sizeof init, cudaMemcpyHostToDevice, st);
    bbox_kernel<<<296, 256, 0, st>>>(xdev, s0, n, dimension, mm);
    unsigned long long hm[6];
    e = cudaMemcpyAsync(hm, mm, sizeof hm, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail_here(WLSQM_E_CUDA, cudaGetErrorString(e));
    double ext[3] = {0, 0, 0};
    GridView& v = g->v;
    v.dim = dimension; v.n = n;
    int deff = 0;
    double vol = 1.0;
    for (int d = 0; d < 3; ++d) {
        v.lo[d] = 0.0; v.dims[d] = 1;
        if (d < dimension) {
            const double lo = dec(hm[d]), hi = dec(hm[3 + d]);
            if (!(lo <= hi)) return fail_here(WLSQM_E_VALUE, "the point set has no finite coordinates");
            v.lo[d] = lo;
            ext[d] = hi - lo;
            if (ext[d] > 0.0) { vol *= ext[d]; ++deff; }
        }
    }
    const double ppc = 2.0;                                       // target points per cell
    double h = 1.0;
    if (deff > 0) {
        h = std::pow(vol / std::max(1.0, (double)n / ppc), 1.0 / deff);
        // (a product of huge finite extents overflows: without this check the loop below never ends)
        if (!std::isfinite(vol) || !std::isfinite(h) || !(h > 0.0))
            return fail_here(WLSQM_E_VALUE, "the extent of the point set is too large for a search grid (overflow)");
        for (int guard = 0;; ++guard) {
            if (guard > 4096) return fail_here(WLSQM_E_VALUE, "no cell size found for the search grid");
            double total = 1.0;
            bool ok = true;
            for (int d = 0; d < dimension; ++d) {
                const double c = std::floor(ext[d] / h) + 1.0;
                if (c > 1048576.0) ok = false;
                total *= c;
            }
            if (ok && total <= std::max(64.0, 4.0 * (double)n) && total < 1.0e9) break;
            h *= 1.25;
        }
    }
    v.h = h; v.inv_h = 1.0 / h;
    long long ncells = 1;
    for (int d = 0; d < dimension; ++d) {
        v.dims[d] = (int)std::floor(ext[d] / h) + 1;
        ncells *= v.dims[d];
    }
    g->ncells = ncells;

    // ---- cell ids, stable sort by cell, start offsets ------------------------------------------------------
    bool okm = dev_alloc((void**)&cid, (size_t)n * 4) == cudaSuccess && dev_alloc((void**)&idx, (size_t)n * 4) == cudaSuccess &&
               dev_alloc((void**)&cid_s, (size_t)n * 4) == cudaSuccess && dev_alloc((void**)&counts, (size_t)(ncells + 1) * 4) == cudaSuccess &&
               dev_alloc((void**)&g->cell_start, (size_t)(ncells + 1) * 4) == cudaSuccess &&
               dev_alloc((void**)&g->sorted_idx, (size_t)n * 4) == cudaSuccess &&
               dev_alloc((void**)&g->sorted_x, (size_t)n * dimension * 8) == cudaSuccess;
    if (!okm) return fail_here(WLSQM_E_MEMORY, "cudaMalloc failed (grid)");
    g->bytes = (ncells + 1) * 4 + n * 4 + n * dimension * 8;
    cudaMemsetAsync(counts, 0, (size_t)(ncells + 1) * 4, st);
    const unsigned nb = (unsigned)((n + 255) / 256);
    cell_id_kernel<<<nb, 256, 0, st>>>(v, xdev, s0, cid, idx, counts);
    size_t tb1 = 0, tb2 = 0;
    int bits = 1;
    while ((1LL << bits) < ncells) ++bits;
    cub::DeviceRadixSort::SortPairs(nullptr, tb1, cid, cid_s, idx, g->sorted_idx, (int)n, 0, bits, st);
    cub::DeviceScan::ExclusiveSum(nullptr, tb2, counts, g->cell_start, (int)(ncells + 1), st);
    if (dev_alloc((void**)&tmp, std::max(tb1, tb2) + 16) != cudaSuccess) return fail_here(WLSQM_E_MEMORY, "cudaMalloc failed (sort)");
    size_t tb = std::max(tb1, tb2) + 16;
    cub::DeviceRadixSort::SortPairs(tmp, tb, cid, cid_s, idx, g->sorted_idx, (int)n, 0, bits, st);
    tb = std::max(tb1, tb2) + 16;
    cub::DeviceScan::ExclusiveSum(tmp, tb, counts, g->cell_start, (int)(ncells + 1), st);
    gather_sorted_kernel<<<(unsigned)((n * dimension + 255) / 256), 256, 0, st>>>(n, dimension, xdev, s0, g->sorted_idx, g->sorted_x);
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail_here(WLSQM_E_CUDA, cudaGetErrorString(e));
    cleanup();
    v.cell_start = g->cell_start; v.sorted_idx = g->sorted_idx; v.sorted_x = g->sorted_x;
    *out = g;
    return WLSQM_OK;
}

int wlsqm_grid_knn(wlsqm_grid_t* g, const double* xq, int64_t xq_s0, int64_t nq, int k, int exclude_self, int32_t* idx32,
                   int64_t* idx64, double* d2) {
    if (!g) return gfail(WLSQM_E_VALUE, "NULL grid");
    if (k < 1 || k > 128) return gfail(WLSQM_E_VALUE, "k must be between 1 and 128");
    if (!xq) nq = g->n;
    if (nq == 0) return WLSQM_OK;
    if (!idx32 && !idx64 && !d2) return gfail(WLSQM_E_VALUE, "no output array given");
    GCU(cudaSetDevice(g->device));
    cudaStream_t st = g->stream;
    // queries / freshly allocated output tensors of the caller: order after what is queued on the caller's stream
    if (order_after_caller(st) != cudaSuccess) { cudaGetLastError(); cudaStreamSynchronize(caller_stream()); }
    const size_t cnt = (size_t)nq * k;
    // host arrays are staged
    double* xqd = nullptr;
    int32_t* o32 = idx32; int64_t* o64 = idx64; double* od2 = d2;
    void *b32 = nullptr, *b64 = nullptr, *bd2 = nullptr;
    auto done = [&](int rc) { dev_free(xqd); dev_free(b32); dev_free(b64); dev_free(bd2); return rc; };
    const double* xqv = xq;
    long long s0 = xq_s0;
    if (xq && !is_dev(xq)) {
        if (dev_alloc((void**)&xqd, (size_t)nq * g->dim * 8) != cudaSuccess) return done(gfail(WLSQM_E_MEMORY, "cudaMalloc failed (queries)"));
        cudaError_t ec = cudaMemcpy2DAsync(xqd, (size_t)g->dim * 8, xq, (size_t)xq_s0 * 8, (size_t)g->dim * 8, (size_t)nq, cudaMemcpyHostToDevice, st);
        if (ec != cudaSuccess) return done(gfail(WLSQM_E_CUDA, cudaGetErrorString(ec)));
        xqv = xqd; s0 = g->dim;
    }
    if (idx32 && !is_dev(idx32)) { if (dev_alloc((void**)&b32, cnt * 4) != cudaSuccess) return done(gfail(WLSQM_E_MEMORY, "cudaMalloc failed")); o32 = (int32_t*)b32; }
    if (idx64 && !is_dev(idx64)) { if (dev_alloc((void**)&b64, cnt * 8) != cudaSuccess) return done(gfail(WLSQM_E_MEMORY, "cudaMalloc failed")); o64 = (int64_t*)b64; }
    if (d2 && !is_dev(d2)) { if (dev_alloc((void**)&bd2, cnt * 8) != cudaSuccess) return done(gfail(WLSQM_E_MEMORY, "cudaMalloc failed")); od2 = (double*)bd2; }
    cudaError_t e;
    if (g->dim == 1) e = launch_knn_d<1>(g->v, xqv, s0, nq, k, exclude_self, o32, o64, od2, st);
    else if (g->dim == 2) e = launch_knn_d<2>(g->v, xqv, s0, nq, k, exclude_self, o32, o64, od2, st);
    else e = launch_knn_d<3>(g->v, xqv, s0, nq, k, exclude_self, o32, o64, od2, st);
    if (e != cudaSuccess) return done(gfail(WLSQM_E_CUDA, cudaGetErrorString(e)));
    if (b32) cudaMemcpyAsync(idx32, b32, cnt * 4, cudaMemcpyDeviceToHost, st);
    if (b64) cudaMemcpyAsync(idx64, b64, cnt * 8, cudaMemcpyDeviceToHost, st);
    if (bd2) cudaMemcpyAsync(d2, bd2, cnt * 8, cudaMemcpyDeviceToHost, st);
    e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return done(gfail(WLSQM_E_CUDA, cudaGetErrorString(e)));
    return done(WLSQM_OK);
}

}  // extern "C"

namespace {

// The device-side inputs of a ball call: queries (host ones staged), radii (host ones staged densely), the error flag.
struct BallInputs {
    BallArgs a{};
    double* xqd = nullptr;
    double* rd = nullptr;
    int* bad = nullptr;
    cudaStream_t st = nullptr;
    ~BallInputs() {
        if (st) cudaStreamSynchronize(st);
        dev_free(xqd); dev_free(rd); dev_free(bad);
    }
};

int ball_inputs(wlsqm_grid* g, const double* xq, int64_t xq_s0, int64_t nq, const double* r, int64_t r_s0,
                int exclude_self, int max_k, BallInputs& in) {
    if (!g) return gfail(WLSQM_E_VALUE, "NULL grid");
    if (!r) return gfail(WLSQM_E_VALUE, "r is NULL");
    if (max_k < 0 || max_k > 128) return gfail(WLSQM_E_VALUE, "max_k must be 0 (no cap) or between 1 and 128");
    if (!xq) nq = g->n;
    if (nq < 0 || r_s0 < 0) return gfail(WLSQM_E_VALUE, "nq and r_s0 must not be negative");
    GCU(cudaSetDevice(g->device));
    cudaStream_t st = g->stream;
    in.st = st;
    // queries, radii and freshly allocated outputs of the caller: order after what is queued on the caller's stream
    if (order_after_caller(st) != cudaSuccess) { cudaGetLastError(); cudaStreamSynchronize(caller_stream()); }
    BallArgs& a = in.a;
    a.xq = xq; a.xq_s0 = xq_s0; a.nq = nq; a.r = r; a.r_s0 = r_s0; a.exclude_self = exclude_self;
    if (dev_alloc((void**)&in.bad, 4) != cudaSuccess) return gfail(WLSQM_E_MEMORY, "cudaMalloc failed");
    GCU(cudaMemsetAsync(in.bad, 0, 4, st));
    a.bad = in.bad;
    if (nq == 0) return WLSQM_OK;
    if (xq && !is_dev(xq)) {
        if (dev_alloc((void**)&in.xqd, (size_t)nq * g->dim * 8) != cudaSuccess) return gfail(WLSQM_E_MEMORY, "cudaMalloc failed (queries)");
        GCU(cudaMemcpy2DAsync(in.xqd, (size_t)g->dim * 8, xq, (size_t)xq_s0 * 8, (size_t)g->dim * 8, (size_t)nq, cudaMemcpyHostToDevice, st));
        a.xq = in.xqd; a.xq_s0 = g->dim;
    }
    if (!is_dev(r)) {
        const long long nr = r_s0 ? nq : 1;
        if (dev_alloc((void**)&in.rd, (size_t)nr * 8) != cudaSuccess) return gfail(WLSQM_E_MEMORY, "cudaMalloc failed (radii)");
        GCU(cudaMemcpy2DAsync(in.rd, 8, r, (size_t)std::max<int64_t>(r_s0, 1) * 8, 8, (size_t)nr, cudaMemcpyHostToDevice, st));
        a.r = in.rd; a.r_s0 = r_s0 ? 1 : 0;
    }
    return WLSQM_OK;
}

// after the stream has been synchronised: a negative or NaN radius fails the call
int ball_check_radii(const BallInputs& in) {
    int bad = 0;
    GCU(cudaMemcpyAsync(&bad, in.bad, 4, cudaMemcpyDeviceToHost, in.st));
    GCU(cudaStreamSynchronize(in.st));
    return bad ? gfail(WLSQM_E_VALUE, "r must be >= 0 and not NaN") : WLSQM_OK;
}

}  // namespace

extern "C" {

int wlsqm_grid_ball_count(wlsqm_grid_t* g, const double* xq, int64_t xq_s0, int64_t nq, const double* r, int64_t r_s0,
                          int exclude_self, int max_k, int64_t* rowptr, int32_t* counts, int64_t* nnz) {
    if (!nnz) return gfail(WLSQM_E_VALUE, "nnz is NULL");
    BallInputs in;
    int rc = ball_inputs(g, xq, xq_s0, nq, r, r_s0, exclude_self, max_k, in);
    if (rc != WLSQM_OK) return rc;
    nq = in.a.nq;
    cudaStream_t st = g->stream;
    long long *c64 = nullptr, *rp = nullptr;
    int32_t* c32 = nullptr;
    void* tmp = nullptr;
    const bool rp_dev = is_dev(rowptr), c_dev = is_dev(counts);
    auto done = [&](int code) {
        cudaStreamSynchronize(st);
        dev_free(c64); if (!rp_dev) dev_free(rp); if (!c_dev) dev_free(c32); dev_free(tmp);
        return code;
    };
    if (dev_alloc((void**)&c64, (size_t)(nq + 1) * 8) != cudaSuccess) return done(gfail(WLSQM_E_MEMORY, "cudaMalloc failed"));
    if (rp_dev) rp = (long long*)rowptr;
    else if (dev_alloc((void**)&rp, (size_t)(nq + 1) * 8) != cudaSuccess) return done(gfail(WLSQM_E_MEMORY, "cudaMalloc failed"));
    if (c_dev) c32 = counts;
    else if (counts && nq && dev_alloc((void**)&c32, (size_t)nq * 4) != cudaSuccess) return done(gfail(WLSQM_E_MEMORY, "cudaMalloc failed"));
    cudaError_t e = launch_ball(g->v, in.a, max_k, c64, c32, nullptr, nullptr, nullptr, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(c64 + nq, 0, 8, st);
    // rowptr = exclusive prefix sum of the counts, nq + 1 entries (the last one is nnz)
    size_t tb = 0;
    if (e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(nullptr, tb, c64, rp, (int)(nq + 1), st);
    if (e == cudaSuccess && dev_alloc(&tmp, tb + 16) != cudaSuccess) return done(gfail(WLSQM_E_MEMORY, "cudaMalloc failed (scan)"));
    if (e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(tmp, tb, c64, rp, (int)(nq + 1), st);
    long long total = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&total, rp + nq, 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && rowptr && !rp_dev) e = cudaMemcpyAsync(rowptr, rp, (size_t)(nq + 1) * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && counts && !c_dev && nq) e = cudaMemcpyAsync(counts, c32, (size_t)nq * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return done(gfail(WLSQM_E_CUDA, cudaGetErrorString(e)));
    rc = ball_check_radii(in);
    if (rc != WLSQM_OK) return done(rc);
    *nnz = total;
    return done(WLSQM_OK);
}

int wlsqm_grid_ball_csr(wlsqm_grid_t* g, const double* xq, int64_t xq_s0, int64_t nq, const double* r, int64_t r_s0,
                        int exclude_self, int max_k, int order, const int64_t* rowptr, int32_t* col) {
    if (order != WLSQM_BALL_BY_INDEX && order != WLSQM_BALL_BY_DISTANCE)
        return gfail(WLSQM_E_VALUE, "order must be WLSQM_BALL_BY_INDEX or WLSQM_BALL_BY_DISTANCE");
    if (!rowptr) return gfail(WLSQM_E_VALUE, "rowptr is NULL");
    BallInputs in;
    int rc = ball_inputs(g, xq, xq_s0, nq, r, r_s0, exclude_self, max_k, in);
    if (rc != WLSQM_OK) return rc;
    nq = in.a.nq;
    cudaStream_t st = g->stream;
    const bool rp_dev = is_dev(rowptr), col_dev = is_dev(col);
    long long nnz = 0;
    if (rp_dev) GCU(cudaMemcpyAsync(&nnz, rowptr + nq, 8, cudaMemcpyDeviceToHost, st));
    GCU(cudaStreamSynchronize(st));
    if (!rp_dev) nnz = rowptr[nq];
    if (nnz < 0) return gfail(WLSQM_E_VALUE, "rowptr[nq] is negative");
    if (nnz > 2147483647LL) return gfail(WLSQM_E_VALUE, "more than 2^31 - 1 entries in one call: split the queries");
    if (nnz > 0 && !col) return gfail(WLSQM_E_VALUE, "col is NULL");
    // device views of rowptr / col: the caller's arrays, or staging buffers owned (and freed) here
    int64_t* rp = rp_dev ? (int64_t*)rowptr : nullptr;
    int32_t *cd = col_dev ? col : nullptr, *c1 = nullptr, *c2 = nullptr;
    double *d1 = nullptr, *d2 = nullptr;
    void* tmp = nullptr;
    auto done = [&](int code) {
        cudaStreamSynchronize(st);
        if (!rp_dev) dev_free(rp);
        if (!col_dev) dev_free(cd);
        dev_free(c1); dev_free(c2); dev_free(d1); dev_free(d2); dev_free(tmp);
        return code;
    };
    auto alloc = [&](void** p, size_t bytes) { return dev_alloc(p, std::max<size_t>(bytes, 16)) == cudaSuccess; };
    if (!rp_dev) {
        if (!alloc((void**)&rp, (size_t)(nq + 1) * 8)) return done(gfail(WLSQM_E_MEMORY, "cudaMalloc failed"));
        const cudaError_t ec = cudaMemcpyAsync(rp, rowptr, (size_t)(nq + 1) * 8, cudaMemcpyHostToDevice, st);
        if (ec != cudaSuccess) return done(gfail(WLSQM_E_CUDA, cudaGetErrorString(ec)));
    }
    if (!col_dev && !alloc((void**)&cd, (size_t)nnz * 4)) return done(gfail(WLSQM_E_MEMORY, "cudaMalloc failed"));
    const bool by_dist = order == WLSQM_BALL_BY_DISTANCE;
    // The fill leaves each row in cell order (uncapped) or in (d2, index) order (capped).  Rows are then sorted by
    // index; for the distance order of the uncapped rows, by index first and then stably by d2.
    const bool sorted_already = max_k > 0 && by_dist;
    if (!sorted_already && !alloc((void**)&c1, (size_t)nnz * 4)) return done(gfail(WLSQM_E_MEMORY, "cudaMalloc failed"));
    const bool with_d2 = max_k == 0 && by_dist;
    if (with_d2 && !(alloc((void**)&c2, (size_t)nnz * 4) && alloc((void**)&d1, (size_t)nnz * 8) &&
                     alloc((void**)&d2, (size_t)nnz * 8)))
        return done(gfail(WLSQM_E_MEMORY, "cudaMalloc failed"));
    cudaError_t e = launch_ball(g->v, in.a, max_k, nullptr, nullptr, rp, sorted_already ? cd : c1, d1, st);
    const int n_items = (int)nnz, n_seg = (int)nq;
    if (e == cudaSuccess && !sorted_already && nnz > 0) {
        size_t tb = 0;
        if (with_d2) {
            size_t tb2 = 0;
            e = cub::DeviceSegmentedSort::SortPairs(nullptr, tb, c1, c2, d1, d2, n_items, n_seg, rp, rp + 1, st);
            if (e == cudaSuccess) e = cub::DeviceSegmentedSort::StableSortPairs(nullptr, tb2, d2, d1, c2, cd, n_items, n_seg, rp, rp + 1, st);
            tb = std::max(tb, tb2);
        } else {
            e = cub::DeviceSegmentedSort::SortKeys(nullptr, tb, c1, cd, n_items, n_seg, rp, rp + 1, st);
        }
        if (e == cudaSuccess && !alloc(&tmp, tb)) return done(gfail(WLSQM_E_MEMORY, "cudaMalloc failed (sort)"));
        if (e == cudaSuccess && with_d2) {
            e = cub::DeviceSegmentedSort::SortPairs(tmp, tb, c1, c2, d1, d2, n_items, n_seg, rp, rp + 1, st);
            if (e == cudaSuccess) e = cub::DeviceSegmentedSort::StableSortPairs(tmp, tb, d2, d1, c2, cd, n_items, n_seg, rp, rp + 1, st);
        } else if (e == cudaSuccess) {
            e = cub::DeviceSegmentedSort::SortKeys(tmp, tb, c1, cd, n_items, n_seg, rp, rp + 1, st);
        }
    }
    if (e == cudaSuccess && !col_dev && nnz > 0) e = cudaMemcpyAsync(col, cd, (size_t)nnz * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return done(gfail(WLSQM_E_CUDA, cudaGetErrorString(e)));
    rc = ball_check_radii(in);
    return done(rc);
}

int wlsqm_grid_info(wlsqm_grid_t* g, int64_t* ncells, double* cell_size, int64_t* bytes) {
    if (!g) return gfail(WLSQM_E_VALUE, "NULL grid");
    if (ncells) *ncells = g->ncells;
    if (cell_size) *cell_size = g->v.h;
    if (bytes) *bytes = g->bytes;
    return WLSQM_OK;
}

}  // extern "C"
