// wlsqm_solve_common.cuh -- the warp GEMV and the ALGO_ITERATIVE refinement of the solve kernels, shared by
// wlsqm_solve.cu (one field per pass) and wlsqm_solve_fields.cu (several fields per pass, which must reproduce its sums
// bit for bit).
#pragma once
#include "wlsqm_common.cuh"
#include "wlsqm_kernels.h"

namespace wlsqm {

// Geometry of the grouped warp GEMV for a case with nr unknowns: the 32 lanes form G = 32/W groups of
// W lanes (W = smallest power of two >= nr, capped at 32); lane = g*W + j.
struct Groups {
    int lw;   // log2(W)
    int W, G, g, j;
};
__device__ __forceinline__ Groups make_groups(int nr, int lane) {
    Groups r;
    r.lw = nr <= 1 ? 0 : (nr > 16 ? 5 : 32 - __clz(nr - 1));
    r.W = 1 << r.lw;
    r.G = 32 >> r.lw;
    r.g = lane >> r.lw;
    r.j = lane & (r.W - 1);
    return r;
}

// shared-memory load on a 32-bit shared address (explicit state space: one LDS, no generic addressing)
__device__ __forceinline__ double lds_f64(uint32_t addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr) : "memory");
    return v;
}

// out[j] = sum_q op[q*nr + j] * v[q], q < n, for one warp.  Group g takes the rows q = g, g+G, ... so that
// one shared-memory wavefront reads G consecutive operator rows (conflict free).  Batches of four rows:
// eight loads are issued before the four independent FMA chains consume them.  A xor-butterfly over the
// groups leaves the total for reduced DOF j in every lane with (lane & (W-1)) == j.
// nr > 32 (3D order 4 with < 3 knowns): lanes also own row j + 32, returned in `hi`.
// op_s / v_s are 32-bit shared-memory addresses.
template <int LW, bool COMPACT>
__device__ __forceinline__ void warp_matvec_t(uint32_t op_s, uint32_t v_s, int n, int nr, int lane, double& lo,
                                              double& hi) {
    constexpr int W = 1 << LW, G = 32 >> LW;
    const int g = lane >> LW, j = lane & (W - 1);
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    hi = 0.0;
    if (j < nr) {
        const uint32_t sp = (uint32_t)(G * nr) * 8u, sp2 = 2u * sp, sp3 = 3u * sp;
        uint32_t pa = op_s + (uint32_t)(g * nr + j) * 8u;
        uint32_t va = v_s + (uint32_t)g * 8u;
        int cnt = (n - g + G - 1) / G;      // rows of this group
        for (; cnt >= 4; cnt -= 4) {
            const double x0 = lds_f64(pa), x1 = lds_f64(pa + sp), x2 = lds_f64(pa + sp2), x3 = lds_f64(pa + sp3);
            double y0, y1, y2, y3;
            if constexpr (G == 1) {       // one group: the four vector entries are consecutive -> two broadcast LDS.128
                asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(y0), "=d"(y1) : "r"(va) : "memory");
                asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(y2), "=d"(y3) : "r"(va + 16u) : "memory");
            } else {
                y0 = lds_f64(va); y1 = lds_f64(va + G * 8); y2 = lds_f64(va + 2 * G * 8); y3 = lds_f64(va + 3 * G * 8);
            }
            a0 = fma(x0, y0, a0);
            a1 = fma(x1, y1, a1);
            a2 = fma(x2, y2, a2);
            a3 = fma(x3, y3, a3);
            pa += 4u * sp;
            va += 4 * G * 8;
        }
        if (cnt >= 2) {
            const double x0 = lds_f64(pa), x1 = lds_f64(pa + sp);
            const double y0 = lds_f64(va), y1 = lds_f64(va + G * 8);
            a0 = fma(x0, y0, a0);
            a1 = fma(x1, y1, a1);
            pa += sp2;
            va += 2 * G * 8;
            cnt -= 2;
        }
        if (cnt > 0) a2 = fma(lds_f64(pa), lds_f64(va), a2);
    }
    if (LW == 5 && nr > 32) {
        // columns 32 .. nr-1 (at most three): every lane takes the rows q = lane, lane + 32, ... of those
        // columns; the partial sums are reduced across the warp and column 32 + t ends up in lane t
        double h0 = 0.0, h1 = 0.0, h2 = 0.0;
        const uint32_t rs8 = (uint32_t)nr * 8u;
        uint32_t qa = op_s + (uint32_t)lane * rs8 + 256u, wa = v_s + (uint32_t)lane * 8u;
        for (int q = lane; q < n; q += 32) {
            const double y = lds_f64(wa);
            h0 = fma(lds_f64(qa), y, h0);
            if (nr > 33) h1 = fma(lds_f64(qa + 8u), y, h1);
            if (nr > 34) h2 = fma(lds_f64(qa + 16u), y, h2);
            qa += 32u * rs8;
            wa += 256u;
        }
        if (nr == 33 || !COMPACT) {
            // (ALGO_BASIC applies the operator once per case and waits on this result: three independent butterflies have
            // the shorter dependency chain; the refinement loop applies it four times and is bound by instruction issue)
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                h0 += __shfl_xor_sync(0xffffffffu, h0, off);
                if (nr > 33) h1 += __shfl_xor_sync(0xffffffffu, h1, off);
                if (nr > 34) h2 += __shfl_xor_sync(0xffffffffu, h2, off);
            }
            hi = lane == 0 ? h0 : (lane == 1 ? h1 : h2);
        } else {
            // two or three sums at once: the first exchange halves the data instead of doubling the shuffles -- the lower
            // 16 lanes go on with column 32, the upper 16 with column 33 (and, for 35 unknowns, the second exchange
            // leaves lanes 8-15 with column 34): 6 / 7 shuffles per application instead of 10 / 15
            const bool up = (lane & 16) != 0;
            double v = (up ? h1 : h0) + __shfl_xor_sync(0xffffffffu, up ? h0 : h1, 16);
            if (nr > 34) {
                const double w = (up ? 0.0 : h2) + __shfl_xor_sync(0xffffffffu, up ? h2 : 0.0, 16);   // lanes 0-15: column 34
                const bool up8 = (lane & 8) != 0;
                v = (up8 ? w : v) + __shfl_xor_sync(0xffffffffu, up8 ? v : w, 8);
            } else {
                v += __shfl_xor_sync(0xffffffffu, v, 8);
            }
#pragma unroll
            for (int off = 4; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
            // column 32 sits in lanes 0-7, column 33 in lanes 16-23, column 34 in lanes 8-15: column 32 + t to lane t
            hi = __shfl_sync(0xffffffffu, v, lane == 1 ? 16 : (lane == 2 ? 8 : 0));
        }
    }
    lo = (a0 + a1) + (a2 + a3);
#pragma unroll
    for (int off = W; off < 32; off <<= 1) lo += __shfl_xor_sync(0xffffffffu, lo, off);
}

template <bool COMPACT>
__device__ __forceinline__ void warp_matvec(uint32_t op_s, uint32_t v_s, int n, int nr, const Groups& gr, int lane,
                                            double& lo, double& hi) {
    switch (gr.lw) {   // warp-uniform
        case 0: warp_matvec_t<0, COMPACT>(op_s, v_s, n, nr, lane, lo, hi); break;
        case 1: warp_matvec_t<1, COMPACT>(op_s, v_s, n, nr, lane, lo, hi); break;
        case 2: warp_matvec_t<2, COMPACT>(op_s, v_s, n, nr, lane, lo, hi); break;
        case 3: warp_matvec_t<3, COMPACT>(op_s, v_s, n, nr, lane, lo, hi); break;
        case 4: warp_matvec_t<4, COMPACT>(op_s, v_s, n, nr, lane, lo, hi); break;
        default: warp_matvec_t<5, COMPACT>(op_s, v_s, n, nr, lane, lo, hi); break;
    }
}

// value of reduced DOF j for original slot o held by this lane (every lane must call it)
__device__ __forceinline__ double fetch_reduced(double lo, double hi, int j) {
    const double vlo = __shfl_sync(0xffffffffu, lo, j & 31);
    const double vhi = __shfl_sync(0xffffffffu, hi, j & 31);
    return j < 32 ? vlo : vhi;
}

// ALGO_ITERATIVE refinement of one case against the data (impl.pyx:1010-1083), with the operator block resident at op_s:
// fis holds the current solution (known slots included), fext the data, rs receives the residuals.  v0 / v1 are this
// lane's slots lane and lane + 32 (updated in place); returns the reference's iteration count.
template <int DIM>
__device__ __forceinline__ int refine_case(const SolveParams& P, long long c, int no, int nk, int nr, const Groups& gr,
                                           int lane, double* fis, const double* xks, const double* fext, double* rs,
                                           uint32_t rs_u32, uint32_t op_s, bool unk0, bool unk1, int j0, int j1,
                                           double& v0, double& v1) {
    int it;
    double xi0 = P.xi[c * P.xi_s0], xi1 = 0.0, xi2 = 0.0;
    if (DIM >= 2) xi1 = P.xi[c * P.xi_s0 + 1];
    if (DIM >= 3) xi2 = P.xi[c * P.xi_s0 + 2];
    double prev = -1.0;
    bool broke = false;
    const bool full_model = no == max_no<DIM>();     // (warp-uniform) order 4: no test per coefficient
    for (it = 0; it < P.max_iter; ++it) {
        double nrm = 0.0;
        if (DIM == 3 && nk > 32) {
            // more neighbours than lanes: a lane evaluates the model at its two neighbours k and k + 32 together
            // (coefficients loaded once, two independent Horner chains).  3D only: the 1D / 2D instantiations run
            // 24 warps per SM at 80 registers and have none to spare for the second chain.
            for (int k = lane; k < nk; k += 64) {
                const int k1 = k + 32;
                const bool has1 = k1 < nk;
                const int kb = has1 ? k1 : k;
                const double dx0 = xks[k * DIM] - xi0, dx1 = xks[kb * DIM] - xi0;
                const double dy0 = DIM >= 2 ? xks[k * DIM + (DIM >= 2 ? 1 : 0)] - xi1 : 0.0;
                const double dy1 = DIM >= 2 ? xks[kb * DIM + (DIM >= 2 ? 1 : 0)] - xi1 : 0.0;
                const double dz0 = DIM >= 3 ? xks[k * DIM + (DIM >= 3 ? 2 : 0)] - xi2 : 0.0;
                const double dz1 = DIM >= 3 ? xks[kb * DIM + (DIM >= 3 ? 2 : 0)] - xi2 : 0.0;
                double m0, m1;
                if (full_model) eval_taylor_nested2<DIM, true>(no, fis, dx0, dy0, dz0, dx1, dy1, dz1, m0, m1);
                else eval_taylor_nested2<DIM, false>(no, fis, dx0, dy0, dz0, dx1, dy1, dz1, m0, m1);
                const double r0 = fext[k] - m0;
                rs[k] = r0;
                const double a0 = fabs(r0);
                nrm = a0 > nrm ? a0 : nrm;          // `if tmp > norm` (impl.pyx:1037-1041)
                if (has1) {
                    const double r1 = fext[k1] - m1;
                    rs[k1] = r1;
                    const double a1 = fabs(r1);
                    nrm = a1 > nrm ? a1 : nrm;
                }
            }
        } else {
            for (int k = lane; k < nk; k += 32) {
                const double dx = xks[k * DIM] - xi0;
                const double dy = DIM >= 2 ? xks[k * DIM + (DIM >= 2 ? 1 : 0)] - xi1 : 0.0;
                const double dz = DIM >= 3 ? xks[k * DIM + (DIM >= 3 ? 2 : 0)] - xi2 : 0.0;
                const double r = fext[k] - (full_model ? eval_taylor_nested_full<DIM>(fis, dx, dy, dz)
                                                       : eval_taylor_nested<DIM>(no, fis, dx, dy, dz));
                rs[k] = r;
                const double ar = fabs(r);
                nrm = ar > nrm ? ar : nrm;          // `if tmp > norm` (impl.pyx:1037-1041)
            }
        }
        nrm = warp_max_nonneg(nrm);
        if (nrm == prev) { broke = true; break; }
        prev = nrm;
        __syncwarp();
        if (nr > 0) {
            double lo, hi;
            warp_matvec<true>(op_s, rs_u32, nk, nr, gr, lane, lo, hi);
            const double t0 = fetch_reduced(lo, hi, j0);
            if (unk0) { v0 += t0; fis[lane] = v0; }
            if (no > 32) {
                const double t1 = fetch_reduced(lo, hi, j1);
                if (unk1) { v1 += t1; fis[lane + 32] = v1; }
            }
        }
        __syncwarp();
    }
    // for/else quirk of impl.pyx:1080-1083: a loop that runs to completion reports max_iter,
    // except max_iter <= 0, which reports 1.
    if (!broke) it = P.max_iter > 0 ? P.max_iter : 1;
    return it;
}

}  // namespace wlsqm
