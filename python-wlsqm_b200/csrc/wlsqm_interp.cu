// wlsqm_interp.cu -- K3: evaluate fitted local models (or any of their derivatives) at query points.
//
// Replaces
//   interpolate_{1,2,3}D / interpolate_nD  wlsqm/fitter/interp.pyx:860-937 / 670-846 / 274-655 / 252-258
//   taylor_* / general_*                   wlsqm/fitter/polyeval.pyx:82-1000
//   expert_interpolate_nearest             wlsqm/fitter/expert.pyx:874-895   (the prange over queries)
//   interpolate_fit                        wlsqm/fitter/interp.pyx:34-143    (single model, I == nullptr)
//
// The model is  f(x) = sum_s fi[s] dx^a dy^b dz^c / (a! b! c!)  with fi[s] the derivative values at the origin.
//
// One derivative slot D = (p,q,r) (the reference's interface): the reference hard-codes, per (dimension,
// derivative), a table that shifts coefficients into a scratch polynomial `fi2` and evaluates that with a nested
// Horner form.  Here the same nested form is generated from the compile-time slot exponent tables,
//   d^D f = sum_{c>=r} dz^(c-r)/(c-r)! sum_{b>=q} dy^(b-q)/(b-q)! sum_{a>=p} fi[a,b,c] dx^(a-p)/(a-p)!,
// each sum as  u0 + h/1 (u1 + h/2 (u2 + h/3 (u3 + ...))), and only the coefficients that D needs are loaded.
// A derivative slot >= no gives 0, as interp.pyx:690-694.
//
// All slots in one pass (WLSQM_DIFF_ALL, extension): every derivative of the model at the query is the Taylor
// shift of the coefficient array, done in place, axis by axis (u_i += h/(i+1) u_{i+1}, repeated): 2D order 4 costs
// 40 FMAs and no registers beyond the 15 coefficients (the term-by-term form needs 70 FMAs and 45 live values).
//
// One thread per query, INTERP_Q queries per thread with their index and coordinate loads issued together.
// WLSQM_DIFF_ALL with dense uniform rows: the warp's 32 x no results are transposed through shared memory so
// that the global stores are contiguous.
#include <cstdlib>
#include <type_traits>
#include "wlsqm_common.cuh"
#include "wlsqm_kernels.h"
#include "wlsqm_grid.h"

namespace wlsqm {

constexpr int INTERP_THREADS = 256;
constexpr int INTERP_Q = 4;        // queries per thread (all slots); the one-slot kernels in 1D / 2D take 2, see launch_interp_m

// ALL = every derivative slot (WLSQM_DIFF_ALL); STAGE = transpose the warp's results through shared memory.
// Each thread owns INTERP_Q queries, blockDim apart (coalesced), and issues their index and coordinate loads
// together before the dependent model-row loads: the kernel is bound by load latency, not by arithmetic.
template <int DIM, bool ALL, bool STAGE, int MINB, int Q>
__global__ void __launch_bounds__(INTERP_THREADS, MINB) interpolate_kernel(InterpParams P) {
    constexpr int NO = max_no<DIM>();
    extern __shared__ __align__(16) double stage[];     // STAGE: [warps][32 * no]
    const long long base = (long long)blockIdx.x * (blockDim.x * Q) + threadIdx.x;
    long long idx[Q];
    double xq[Q][DIM];
#pragma unroll
    for (int j = 0; j < Q; ++j) {
        const long long m = base + (long long)j * blockDim.x;
        const long long mm = m < P.nx ? m : P.nx - 1;
        idx[j] = P.I ? P.I[mm] : 0;
#pragma unroll
        for (int d = 0; d < DIM; ++d) xq[j][d] = P.x[mm * P.x_s0 + d];
    }
    // the model rows of all Q queries are requested before the first one is used: the chain index -> row is the
    // latency that bounds this kernel, and an in-order thread would otherwise pay it once per query
#pragma unroll
    for (int j = 0; j < Q; ++j) {
        const bool bad = P.nmodels > 0 && (idx[j] < 0 || idx[j] >= P.nmodels);
        const double* fg = P.fi + (bad ? 0 : idx[j]) * P.fi_s0;
        asm volatile("prefetch.global.L1 [%0];" ::"l"(fg));
        asm volatile("prefetch.global.L1 [%0];" ::"l"(P.xi + (bad ? 0 : idx[j]) * P.xi_s0));
        if (DIM >= 2) asm volatile("prefetch.global.L1 [%0];" ::"l"(fg + (DIM == 2 ? 14 : 16)));
        if (DIM >= 3) asm volatile("prefetch.global.L1 [%0];" ::"l"(fg + 34));
    }
#pragma unroll
    for (int j = 0; j < Q; ++j) {
        const long long m = base + (long long)j * blockDim.x;
        const bool live = m < P.nx;
        // "no neighbour found" (index == number of models, cKDTree's convention for a NaN query) -> NaN
        const bool bad = P.nmodels > 0 && (idx[j] < 0 || idx[j] >= P.nmodels);
        const long long i = bad ? 0 : idx[j];
        const int order = P.order ? (int)P.order[i] : P.order_uniform;
        const int no = dofs_of<DIM>(order);
        const double* xo = P.xi + i * P.xi_s0;
        const double dx = xq[j][0] - xo[0];
        const double dy = DIM >= 2 ? xq[j][DIM >= 2 ? 1 : 0] - xo[DIM >= 2 ? 1 : 0] : 0.0;
        const double dz = DIM >= 3 ? xq[j][DIM >= 3 ? 2 : 0] - xo[DIM >= 3 ? 2 : 0] : 0.0;
        const double* fg = P.fi + i * P.fi_s0;
        if constexpr (!ALL) {
            const Steps hx = steps_of(dx), hy = steps_of(dy), hz = steps_of(dz);
            double v = 0.0;
            static_for<0, NO>([&](auto I) {
                constexpr int D = decltype(I)::value;
                if (P.diff == D) v = eval_diff<DIM, D>(fg, no, hx, hy, hz);     // grid-uniform branch
            });
            if (live) st_stream(P.out + m, bad ? __longlong_as_double(0x7ff8000000000000LL) : v);
        } else {
            // extension: every derivative slot of the model in one pass, out[m][0..no)
            double u[NO];
#pragma unroll
            for (int s = 0; s < NO; ++s) u[s] = s < no ? __ldg(fg + s) : 0.0;
            taylor_shift<DIM, 0>(u, dx);
            if constexpr (DIM >= 2) taylor_shift<DIM, 1>(u, dy);
            if constexpr (DIM >= 3) taylor_shift<DIM, 2>(u, dz);
            if (bad) {
#pragma unroll
                for (int s = 0; s < NO; ++s) u[s] = __longlong_as_double(0x7ff8000000000000LL);
            }
            if constexpr (STAGE) {
                // uniform model size and dense rows: transpose through shared memory, then contiguous stores
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
                double* o = P.out + m0 * nno;
                for (int t = lane; t < 32 * nno && t < left; t += 32) st_stream(o + t, st[t]);
            } else if (live) {
                double* o = P.out + m * P.out_s0;
#pragma unroll
                for (int d = 0; d < NO; ++d)
                    if (d < no) st_stream(o + d, u[d]);
            }
        }
    }
}

// mode='continuous' (expert_interpolate_continuous, wlsqm/fitter/expert.pyx:898-985): weighted average of every
// local model whose origin lies within r of the query, weights (1 - sqrt(d2 / r2))^2 (alpha = 0, beta = 1,
// expert.pyx:45-46).  The reference finds the models with cKDTree.query_ball_tree and loops in Python; here one
// thread per query walks the cells of the model-origin grid that intersect its ball and evaluates on the fly.
template <int DIM>
__global__ void __launch_bounds__(128) continuous_kernel(InterpParams P, GridView g, double r) {
    constexpr int NO = max_no<DIM>();
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
    double acc = 0.0, sum_w = 0.0;
    for (int cz = c0[2]; cz <= c1[2]; ++cz)
        for (int cy = c0[1]; cy <= c1[1]; ++cy) {
            const long long row = ((long long)cz * g.dims[1] + cy) * g.dims[0];
            const int p1 = g.cell_start[row + c1[0] + 1];
            for (int p = g.cell_start[row + c0[0]]; p < p1; ++p) {     // the cells of one x-row are contiguous
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
                const double* fg = P.fi + i * P.fi_s0;
                const Steps hx = steps_of(dq[0]), hy = steps_of(dq[1]), hz = steps_of(dq[2]);
                double value = 0.0;
                static_for<0, NO>([&](auto I) {
                    constexpr int D = decltype(I)::value;
                    if (P.diff == D) value = eval_diff<DIM, D>(fg, no, hx, hy, hz);
                });
                const double tmp = 1.0 - sqrt(d2 / r2);
                const double w = tmp * tmp;
                acc += w * value;
                sum_w += w;
            }
        }
    P.out[m] = acc / sum_w;     // no model within r: 0/0 = NaN, like the reference
}

cudaError_t launch_interpolate_continuous(const InterpParams& P, const GridView& g, double r, cudaStream_t st) {
    if (P.nx == 0) return cudaSuccess;
    const unsigned blocks = (unsigned)((P.nx + 127) / 128);
    if (P.dim == 1) continuous_kernel<1><<<blocks, 128, 0, st>>>(P, g, r);
    else if (P.dim == 2) continuous_kernel<2><<<blocks, 128, 0, st>>>(P, g, r);
    else continuous_kernel<3><<<blocks, 128, 0, st>>>(P, g, r);
    return cudaGetLastError();
}

template <int DIM, bool ALL, bool STAGE, int MINB, int Q>
static cudaError_t launch_interp_t(const InterpParams& P, size_t smem, cudaStream_t st) {
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(interpolate_kernel<DIM, ALL, STAGE, MINB, Q>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    const long long per_block = (long long)INTERP_THREADS * Q;
    const unsigned blocks = (unsigned)((P.nx + per_block - 1) / per_block);
    interpolate_kernel<DIM, ALL, STAGE, MINB, Q><<<blocks, INTERP_THREADS, smem, st>>>(P);
    return cudaGetLastError();
}

// Resident CTAs per SM the register budget is held to, and queries per thread (WLSQM_INTERP_MINB / WLSQM_INTERP_Q override,
// for tuning).  All slots: 4 queries per thread at 4 CTAs (2 in 3D) -- the Taylor shift holds the whole model in
// registers.  One slot per call (the reference's interface) is a short dependent chain -- query index -> model row -> a
// dozen FMAs -- bound by load latency: TWO queries per thread fit 32 registers without spills, i.e. 8 CTAs = every warp
// slot of the SM (measured, 16M queries 2D: 4 queries x 4 CTAs 0.196 ms, 4 x 6 0.164, 4 x 8 with spills 0.151,
// 2 x 8 0.144 ms; the reference's 15 calls 2.14 -> 1.59 ms = 0.94 of the HBM peak).
template <int DIM, bool ALL, bool STAGE>
static cudaError_t launch_interp_m(const InterpParams& P, size_t smem, cudaStream_t st) {
    static const int forced = [] { const char* v = getenv("WLSQM_INTERP_MINB"); return (v && *v) ? atoi(v) : 0; }();
    static const int forced_q = [] { const char* v = getenv("WLSQM_INTERP_Q"); return (v && *v) ? atoi(v) : 0; }();
    if constexpr (!ALL && DIM < 3) {
        const int minb = forced > 0 ? forced : 8;
        const int q = forced_q > 0 ? forced_q : 2;
        if (q >= 4) {
            if (minb <= 4) return launch_interp_t<DIM, ALL, STAGE, 4, 4>(P, smem, st);
            if (minb <= 6) return launch_interp_t<DIM, ALL, STAGE, 6, 4>(P, smem, st);
            return launch_interp_t<DIM, ALL, STAGE, 8, 4>(P, smem, st);
        }
        if (q == 1) return launch_interp_t<DIM, ALL, STAGE, 8, 1>(P, smem, st);
        if (minb <= 4) return launch_interp_t<DIM, ALL, STAGE, 4, 2>(P, smem, st);
        if (minb <= 6) return launch_interp_t<DIM, ALL, STAGE, 6, 2>(P, smem, st);
        return launch_interp_t<DIM, ALL, STAGE, 8, 2>(P, smem, st);
    } else if constexpr (!ALL) {
        // 3D: 35 coefficients per model; ONE query per thread at 8 CTAs (31 registers, a few spilled words) beats every
        // other point (8M queries, value / highest slot: 4 x 3 CTAs 0.213 / 0.102 ms, 2 x 6 0.151 / 0.087, 1 x 8 0.141 / 0.085)
        const int minb = forced > 0 ? forced : 8;
        const int q = forced_q > 0 ? forced_q : 1;
        if (q >= 4) {
            if (minb <= 2) return launch_interp_t<DIM, ALL, STAGE, 2, 4>(P, smem, st);
            if (minb == 3) return launch_interp_t<DIM, ALL, STAGE, 3, 4>(P, smem, st);
            return launch_interp_t<DIM, ALL, STAGE, 4, 4>(P, smem, st);
        }
        if (q == 1) {
            if (minb <= 5) return launch_interp_t<DIM, ALL, STAGE, 5, 1>(P, smem, st);
            if (minb <= 6) return launch_interp_t<DIM, ALL, STAGE, 6, 1>(P, smem, st);
            return launch_interp_t<DIM, ALL, STAGE, 8, 1>(P, smem, st);
        }
        if (minb <= 2) return launch_interp_t<DIM, ALL, STAGE, 2, 2>(P, smem, st);
        if (minb == 3) return launch_interp_t<DIM, ALL, STAGE, 3, 2>(P, smem, st);
        if (minb == 4) return launch_interp_t<DIM, ALL, STAGE, 4, 2>(P, smem, st);
        if (minb == 5) return launch_interp_t<DIM, ALL, STAGE, 5, 2>(P, smem, st);
        return launch_interp_t<DIM, ALL, STAGE, 6, 2>(P, smem, st);
    } else {
        const int minb = forced > 0 ? forced : (DIM == 3 ? 2 : 4);
        if (minb <= 2) return launch_interp_t<DIM, ALL, STAGE, 2, INTERP_Q>(P, smem, st);
        if (minb == 3) return launch_interp_t<DIM, ALL, STAGE, 3, INTERP_Q>(P, smem, st);
        return launch_interp_t<DIM, ALL, STAGE, 4, INTERP_Q>(P, smem, st);
    }
}

template <int DIM>
static cudaError_t launch_interp_d(const InterpParams& P, size_t smem, cudaStream_t st) {
    if (P.diff >= 0) return launch_interp_m<DIM, false, false>(P, 0, st);
    if (P.stage_no > 0) return launch_interp_m<DIM, true, true>(P, smem, st);
    return launch_interp_m<DIM, true, false>(P, 0, st);
}

cudaError_t launch_interpolate(const InterpParams& Pin, cudaStream_t st) {
    if (Pin.nx == 0) return cudaSuccess;
    InterpParams P = Pin;
    size_t smem = 0;
    if (P.diff < 0 && P.stage_no > 0) smem = (size_t)(INTERP_THREADS / 32) * 32 * P.stage_no * sizeof(double);
    else P.stage_no = 0;
    if (P.dim == 1) return launch_interp_d<1>(P, smem, st);
    if (P.dim == 2) return launch_interp_d<2>(P, smem, st);
    return launch_interp_d<3>(P, smem, st);
}

}  // namespace wlsqm
