// wlsqm_interp_fields.cu -- K3 for several fields on one geometry: evaluate caller-held solutions fi[j] at query points
// (InterpFieldsParams, wlsqm_kernels.h), in nearest and continuous mode.
//
// Field j of the output is bit for bit what interpolate_kernel / continuous_kernel (wlsqm_interp.cu) write when the
// solver's solution copy holds fi[j]: the slots come from the same helpers (eval_diff for one slot, taylor_shift for all
// slots) at the same offsets, and the continuous sums keep continuous_kernel's expression forms and visiting order.
// What a query does once for all fields of a pass instead of once per field: the index and coordinate loads, the origin
// row, the Taylor steps and, in continuous mode, the walk over the model grid (candidates, d2, membership, weight).
//
// Fields per pass: up to 8, register-blocked in the one-slot and continuous kernels; the all-slots kernel holds one
// field's coefficients at a time and only requests the pass's rows together.  How many fields a pass takes is decided
// by interp_fields_per_pass below from the sizes of the call: reading more fields at once multiplies the model-row
// footprint, and where that footprint outgrows L2 the rows that queries share are fetched from DRAM again.
#include <cmath>
#include "wlsqm_common.cuh"
#include "wlsqm_kernels.h"
#include "wlsqm_grid.h"

namespace wlsqm {

constexpr int IF_THREADS = 256;
constexpr int IF_CONT_THREADS = 128;

__device__ __forceinline__ void prefetch_row(const double* fg, int dim) {
    asm volatile("prefetch.global.L1 [%0];" ::"l"(fg));
    if (dim >= 2) asm volatile("prefetch.global.L1 [%0];" ::"l"(fg + (dim == 2 ? 14 : 16)));
    if (dim >= 3) asm volatile("prefetch.global.L1 [%0];" ::"l"(fg + 34));
}

// one slot (P.diff >= 0), FB fields per thread in registers; one query per thread
template <int DIM, int FB>
__global__ void __launch_bounds__(IF_THREADS) interp_fields_kernel(InterpFieldsParams F) {
    constexpr int NO = max_no<DIM>();
    const InterpParams& P = F.P;
    const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= P.nx) return;
    const long long idx = P.I[m];
    double xq[DIM];
#pragma unroll
    for (int d = 0; d < DIM; ++d) xq[d] = P.x[m * P.x_s0 + d];
    const bool bad = idx < 0 || idx >= P.nmodels;
    const long long i = bad ? 0 : idx;
    // the rows of every field of the pass are requested before the first one is used
    asm volatile("prefetch.global.L1 [%0];" ::"l"(P.xi + i * P.xi_s0));
#pragma unroll
    for (int j = 0; j < FB; ++j)
        if (j < F.nf) prefetch_row(P.fi + j * F.fi_sf + i * P.fi_s0, DIM);
    const int order = P.order ? (int)P.order[i] : P.order_uniform;
    const int no = dofs_of<DIM>(order);
    const double* xo = P.xi + i * P.xi_s0;
    const double dx = xq[0] - xo[0];
    const double dy = DIM >= 2 ? xq[DIM >= 2 ? 1 : 0] - xo[DIM >= 2 ? 1 : 0] : 0.0;
    const double dz = DIM >= 3 ? xq[DIM >= 3 ? 2 : 0] - xo[DIM >= 3 ? 2 : 0] : 0.0;
    const Steps hx = steps_of(dx), hy = steps_of(dy), hz = steps_of(dz);
    double v[FB];
#pragma unroll
    for (int j = 0; j < FB; ++j) v[j] = 0.0;
    static_for<0, NO>([&](auto I) {
        constexpr int D = decltype(I)::value;
        if (P.diff == D) {     // grid-uniform branch
#pragma unroll
            for (int j = 0; j < FB; ++j)
                if (j < F.nf) v[j] = eval_diff<DIM, D>(P.fi + j * F.fi_sf + i * P.fi_s0, no, hx, hy, hz);
        }
    });
#pragma unroll
    for (int j = 0; j < FB; ++j)
        if (j < F.nf) st_stream(P.out + j * F.out_sf + m * P.out_s0, bad ? __longlong_as_double(0x7ff8000000000000LL) : v[j]);
}

// every slot (WLSQM_DIFF_ALL): out[j][q][0..width), zeros in slots >= no_i.  STAGE: every model has P.stage_no ==
// width DOFs and out_s0 == width, so the warp's 32 rows of a field are contiguous: transposed through shared memory
// (as interpolate_kernel does), then stored with contiguous stores.
template <int DIM, bool STAGE>
__global__ void __launch_bounds__(IF_THREADS) interp_fields_all_kernel(InterpFieldsParams F) {
    constexpr int NO = max_no<DIM>();
    extern __shared__ __align__(16) double stage[];     // STAGE: [warps][32 * no]
    const InterpParams& P = F.P;
    const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = m < P.nx;
    const long long mm = live ? m : P.nx - 1;
    const long long idx = P.I[mm];
    double xq[DIM];
#pragma unroll
    for (int d = 0; d < DIM; ++d) xq[d] = P.x[mm * P.x_s0 + d];
    const bool bad = idx < 0 || idx >= P.nmodels;
    const long long i = bad ? 0 : idx;
    asm volatile("prefetch.global.L1 [%0];" ::"l"(P.xi + i * P.xi_s0));
    for (int j = 0; j < F.nf; ++j) prefetch_row(P.fi + j * F.fi_sf + i * P.fi_s0, DIM);
    const int order = P.order ? (int)P.order[i] : P.order_uniform;
    const int no = dofs_of<DIM>(order);
    const double* xo = P.xi + i * P.xi_s0;
    const double dx = xq[0] - xo[0];
    const double dy = DIM >= 2 ? xq[DIM >= 2 ? 1 : 0] - xo[DIM >= 2 ? 1 : 0] : 0.0;
    const double dz = DIM >= 3 ? xq[DIM >= 3 ? 2 : 0] - xo[DIM >= 3 ? 2 : 0] : 0.0;
    const Steps hx = steps_of(dx), hy = steps_of(dy), hz = steps_of(dz);
#pragma unroll 1
    for (int j = 0; j < F.nf; ++j) {
        const double* fg = P.fi + j * F.fi_sf + i * P.fi_s0;
        double u[NO];
#pragma unroll
        for (int s = 0; s < NO; ++s) u[s] = s < no ? __ldg(fg + s) : 0.0;
        taylor_shift<DIM, 0>(u, hx);
        if constexpr (DIM >= 2) taylor_shift<DIM, 1>(u, hy);
        if constexpr (DIM >= 3) taylor_shift<DIM, 2>(u, hz);
        if (bad) {
#pragma unroll
            for (int s = 0; s < NO; ++s) u[s] = __longlong_as_double(0x7ff8000000000000LL);
        }
        double* out = P.out + j * F.out_sf;
        if constexpr (STAGE) {
            const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
            const int nno = P.stage_no;
            double* st = stage + (size_t)warp * 32 * nno;
            __syncwarp();
#pragma unroll
            for (int d = 0; d < NO; ++d)
                if (d < nno) st[lane * nno + d] = u[d];
            __syncwarp();
            const long long m0 = m - lane;                       // first query of this warp
            const long long left = (P.nx - m0) * nno;            // doubles this warp may still write
            double* o = out + m0 * nno;
            for (int t = lane; t < 32 * nno && t < left; t += 32) st_stream(o + t, st[t]);
        } else if (live) {
            double* o = out + m * P.out_s0;
#pragma unroll
            for (int d = 0; d < NO; ++d)
                if (d < F.width) st_stream(o + d, d < no ? u[d] : 0.0);
        }
    }
}

// mode='continuous' for FB fields: continuous_kernel's walk, once per query; per field its own acc with the same
// expression forms and order of visits, then acc / sum_w (no model within r: 0/0 = NaN)
template <int DIM, int FB>
__global__ void __launch_bounds__(IF_CONT_THREADS, 1) continuous_fields_kernel(InterpFieldsParams F, GridView g, double r) {
    constexpr int NO = max_no<DIM>();
    const InterpParams& P = F.P;
    const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= P.nx) return;
    double q[3] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int d = 0; d < DIM; ++d) q[d] = P.x[m * P.x_s0 + d];
    const double r2 = r * r;
    int c0[3] = {0, 0, 0}, c1[3] = {0, 0, 0};
#pragma unroll
    for (int d = 0; d < DIM; ++d) {
        c0[d] = grid_cell_coord(g, d, q[d] - r);
        c1[d] = grid_cell_coord(g, d, q[d] + r);
    }
    double acc[FB], sum_w = 0.0;
#pragma unroll
    for (int j = 0; j < FB; ++j) acc[j] = 0.0;
    for (int cz = c0[2]; cz <= c1[2]; ++cz)
        for (int cy = c0[1]; cy <= c1[1]; ++cy) {
            const long long row = ((long long)cz * g.dims[1] + cy) * g.dims[0];
            const int p1 = g.cell_start[row + c1[0] + 1];
            for (int p = g.cell_start[row + c0[0]]; p < p1; ++p) {
                double d2 = 0.0, dq[3] = {0.0, 0.0, 0.0};
#pragma unroll
                for (int d = 0; d < DIM; ++d) {
                    dq[d] = q[d] - g.sorted_x[(long long)p * DIM + d];
                    d2 += dq[d] * dq[d];
                }
                if (!(d2 <= r2)) continue;
                const long long i = g.sorted_idx[p];
                const int order = P.order ? (int)P.order[i] : P.order_uniform;
                const int no = dofs_of<DIM>(order);
                const Steps hx = steps_of(dq[0]), hy = steps_of(dq[1]), hz = steps_of(dq[2]);
                double value[FB];
#pragma unroll
                for (int j = 0; j < FB; ++j) value[j] = 0.0;
                static_for<0, NO>([&](auto I) {
                    constexpr int D = decltype(I)::value;
                    if (P.diff == D) {
#pragma unroll
                        for (int j = 0; j < FB; ++j)
                            if (j < F.nf) value[j] = eval_diff<DIM, D>(P.fi + j * F.fi_sf + i * P.fi_s0, no, hx, hy, hz);
                    }
                });
                const double tmp = 1.0 - sqrt(d2 / r2);
                const double w = tmp * tmp;
#pragma unroll
                for (int j = 0; j < FB; ++j) acc[j] += w * value[j];
                sum_w += w;
            }
        }
#pragma unroll
    for (int j = 0; j < FB; ++j)
        if (j < F.nf) P.out[j * F.out_sf + m * P.out_s0] = acc[j] / sum_w;
}

// Fields per pass (1, 2, 4 or 8) from a byte model of the DRAM traffic of the whole call, nf fields over nx queries:
//   - every query reads query_bytes once per pass (coordinates and index, or the grid walk) and writes out_bytes per field;
//   - per field it reads rows_per_query model rows of rb bytes (the 32-byte sectors a row of max no doubles spans, averaged
//     over its alignment); A = nx * rows_per_query row reads over U = ncases (1 - exp(-A / ncases)) distinct rows;
//   - a pass of f fields keeps f U rb bytes of rows live.  Within L2 every row comes from DRAM once per field; beyond it
//     (random queries, so no locality to exploit) a repeated read hits with probability L2 / footprint.
// The plan with the fewest bytes wins; ties go to more fields per pass (fewer launches, the latency of a query's
// index -> row chain paid once for more fields).
int interp_fields_per_pass(long long nf, long long ncases, int maxno, long long nx, double rows_per_query,
                           double query_bytes, double out_bytes, long long l2_bytes) {
    if (nf <= 1 || ncases <= 0 || nx <= 0) return 1;
    double rb = 0.0;
    for (int off = 0; off < 32; off += 8) rb += 32.0 * std::ceil((off + 8.0 * maxno) / 32.0) / 4.0;
    const double A = (double)nx * rows_per_query;
    const double U = (double)ncases * -std::expm1(-A / (double)ncases);
    int best_f = 1;
    double best = 0.0;
    for (int f = 1; f <= 8; f *= 2) {
        if (f > 1 && f / 2 >= nf) break;
        const double live = (double)std::min<long long>(f, nf) * U * rb;
        const double hit = live <= (double)l2_bytes ? 1.0 : (double)l2_bytes / live;
        const double rows = U * rb + (A - U) * rb * (1.0 - hit);
        const double passes = (double)((nf + f - 1) / f);
        const double bytes = (double)nf * (rows + (double)nx * out_bytes) + passes * (double)nx * query_bytes;
        if (f == 1 || bytes <= best) { best = bytes; best_f = f; }
    }
    return best_f;
}

// fi rows that are not dense (fields-inner, pitched), copied to dense rows for one pass: dst[j][i][s] = src[j*sf + i*s0 + s]
// for j < nfp, s < maxno.  One thread per element, consecutive threads on consecutive elements of a row.
__global__ void __launch_bounds__(IF_THREADS) compact_rows_kernel(const double* __restrict__ src, long long sf, long long s0,
                                                                   long long n, int maxno, double* __restrict__ dst) {
    const long long per = n * maxno;
    const int j = blockIdx.y;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < per; e += (long long)gridDim.x * blockDim.x) {
        const long long i = e / maxno;
        dst[j * per + e] = __ldg(src + j * sf + i * s0 + (e - i * maxno));
    }
}

cudaError_t launch_compact_rows(const double* src, long long sf, long long s0, int nfp, long long n, int maxno, double* dst,
                                cudaStream_t st) {
    if (nfp == 0 || n == 0) return cudaSuccess;
    const long long per = n * maxno;
    const unsigned bx = (unsigned)std::min<long long>((per + IF_THREADS - 1) / IF_THREADS, 148 * 16);
    compact_rows_kernel<<<dim3(bx, (unsigned)nfp), IF_THREADS, 0, st>>>(src, sf, s0, n, maxno, dst);
    return cudaGetLastError();
}

template <int DIM>
static cudaError_t launch_fields_d(const InterpFieldsParams& F, cudaStream_t st) {
    const InterpParams& P = F.P;
    const unsigned blocks = (unsigned)((P.nx + IF_THREADS - 1) / IF_THREADS);
    if (P.diff >= 0) {
        if (F.nf <= 1) interp_fields_kernel<DIM, 1><<<blocks, IF_THREADS, 0, st>>>(F);
        else if (F.nf <= 2) interp_fields_kernel<DIM, 2><<<blocks, IF_THREADS, 0, st>>>(F);
        else if (F.nf <= 4) interp_fields_kernel<DIM, 4><<<blocks, IF_THREADS, 0, st>>>(F);
        else interp_fields_kernel<DIM, 8><<<blocks, IF_THREADS, 0, st>>>(F);
    } else if (P.stage_no > 0) {
        const size_t smem = (size_t)(IF_THREADS / 32) * 32 * P.stage_no * sizeof(double);
        if (smem > 48 * 1024) {
            const cudaError_t e = cudaFuncSetAttribute(interp_fields_all_kernel<DIM, true>,
                                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        interp_fields_all_kernel<DIM, true><<<blocks, IF_THREADS, smem, st>>>(F);
    } else {
        interp_fields_all_kernel<DIM, false><<<blocks, IF_THREADS, 0, st>>>(F);
    }
    return cudaGetLastError();
}

cudaError_t launch_interpolate_fields(const InterpFieldsParams& F, cudaStream_t st) {
    if (F.P.nx == 0 || F.nf == 0) return cudaSuccess;
    if (F.P.dim == 1) return launch_fields_d<1>(F, st);
    if (F.P.dim == 2) return launch_fields_d<2>(F, st);
    return launch_fields_d<3>(F, st);
}

template <int DIM>
static cudaError_t launch_continuous_fields_d(const InterpFieldsParams& F, const GridView& g, double r, cudaStream_t st) {
    const unsigned blocks = (unsigned)((F.P.nx + IF_CONT_THREADS - 1) / IF_CONT_THREADS);
    if (F.nf <= 1) continuous_fields_kernel<DIM, 1><<<blocks, IF_CONT_THREADS, 0, st>>>(F, g, r);
    else if (F.nf <= 2) continuous_fields_kernel<DIM, 2><<<blocks, IF_CONT_THREADS, 0, st>>>(F, g, r);
    else if (F.nf <= 4) continuous_fields_kernel<DIM, 4><<<blocks, IF_CONT_THREADS, 0, st>>>(F, g, r);
    else continuous_fields_kernel<DIM, 8><<<blocks, IF_CONT_THREADS, 0, st>>>(F, g, r);
    return cudaGetLastError();
}

cudaError_t launch_interpolate_continuous_fields(const InterpFieldsParams& F, const GridView& g, double r, cudaStream_t st) {
    if (F.P.nx == 0 || F.nf == 0) return cudaSuccess;
    if (F.P.dim == 1) return launch_continuous_fields_d<1>(F, g, r, st);
    if (F.P.dim == 2) return launch_continuous_fields_d<2>(F, g, r, st);
    return launch_continuous_fields_d<3>(F, g, r, st);
}

}  // namespace wlsqm
