// wlsqm_solve_fields.cu -- K2 for several fields on one geometry (FieldsParams, wlsqm_kernels.h).
//
// A multi-field time step (velocity components, temperature, concentration) fits every field on the same
// neighbourhoods.  Solved one field at a time, each field streams the whole operator block again: at 2D order 4 with
// k = 30 that is 3600 of the 3960 bytes a case moves.  Here each block is streamed once per pass for all fields of the
// pass; a stage of the ring is [operator | fext of field 0 | ... | fext of field F-1 | xk (ITER)].
//
// Every field keeps exactly the summation order of the kernel that a single-field solve picks (solve_kernel's grouped
// warp GEMV, solve_pack_kernel's sequential column chain, the refinement and its exact-equality exit), so each result is
// bit for bit that solve's; only the reads of the operator elements are shared.  The GEMV and the refinement are
// solve_kernel's own (wlsqm_solve_common.cuh).
#include <type_traits>
#include "wlsqm_common.cuh"
#include "wlsqm_kernels.h"
#include "wlsqm_solve_common.cuh"

namespace wlsqm {

// warp_matvec_t<LW, false> for FB fields at once: each operator element read from shared memory feeds the four FMA
// chains of every field (fields f < nfb; the vector of field f at v_s + f * vstride), so that issue per field and row
// is one vector load and one FMA.
template <int LW, int FB>
__device__ __forceinline__ void warp_matvec_fields_t(uint32_t op_s, uint32_t v_s, uint32_t vstride, int nfb, int n, int nr,
                                                     int lane, double (&lo)[FB], double (&hi)[FB]) {
    constexpr int W = 1 << LW, G = 32 >> LW;
    const int g = lane >> LW, j = lane & (W - 1);
    double a0[FB], a1[FB], a2[FB], a3[FB];
#pragma unroll
    for (int f = 0; f < FB; ++f) { a0[f] = a1[f] = a2[f] = a3[f] = 0.0; hi[f] = 0.0; }
    if (j < nr) {
        const uint32_t sp = (uint32_t)(G * nr) * 8u, sp2 = 2u * sp, sp3 = 3u * sp;
        uint32_t pa = op_s + (uint32_t)(g * nr + j) * 8u;
        uint32_t va = v_s + (uint32_t)g * 8u;
        int cnt = (n - g + G - 1) / G;
        for (; cnt >= 4; cnt -= 4) {
            const double x0 = lds_f64(pa), x1 = lds_f64(pa + sp), x2 = lds_f64(pa + sp2), x3 = lds_f64(pa + sp3);
#pragma unroll
            for (int f = 0; f < FB; ++f) {
                if (f < nfb) {
                    const uint32_t vf = va + (uint32_t)f * vstride;
                    double y0, y1, y2, y3;
                    if constexpr (G == 1) {
                        asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(y0), "=d"(y1) : "r"(vf) : "memory");
                        asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(y2), "=d"(y3) : "r"(vf + 16u) : "memory");
                    } else {
                        y0 = lds_f64(vf); y1 = lds_f64(vf + G * 8); y2 = lds_f64(vf + 2 * G * 8); y3 = lds_f64(vf + 3 * G * 8);
                    }
                    a0[f] = fma(x0, y0, a0[f]);
                    a1[f] = fma(x1, y1, a1[f]);
                    a2[f] = fma(x2, y2, a2[f]);
                    a3[f] = fma(x3, y3, a3[f]);
                }
            }
            pa += 4u * sp;
            va += 4 * G * 8;
        }
        if (cnt >= 2) {
            const double x0 = lds_f64(pa), x1 = lds_f64(pa + sp);
#pragma unroll
            for (int f = 0; f < FB; ++f) {
                if (f < nfb) {
                    const uint32_t vf = va + (uint32_t)f * vstride;
                    a0[f] = fma(x0, lds_f64(vf), a0[f]);
                    a1[f] = fma(x1, lds_f64(vf + G * 8), a1[f]);
                }
            }
            pa += sp2;
            va += 2 * G * 8;
            cnt -= 2;
        }
        if (cnt > 0) {
            const double x0 = lds_f64(pa);
#pragma unroll
            for (int f = 0; f < FB; ++f)
                if (f < nfb) a2[f] = fma(x0, lds_f64(va + (uint32_t)f * vstride), a2[f]);
        }
    }
    if (LW == 5 && nr > 32) {
        // columns 32 .. nr-1: per field as in warp_matvec_t (three independent butterflies)
#pragma unroll
        for (int f = 0; f < FB; ++f) {
            if (f >= nfb) break;
            double h0 = 0.0, h1 = 0.0, h2 = 0.0;
            const uint32_t rs8 = (uint32_t)nr * 8u;
            uint32_t qa = op_s + (uint32_t)lane * rs8 + 256u, wa = v_s + (uint32_t)f * vstride + (uint32_t)lane * 8u;
            for (int q = lane; q < n; q += 32) {
                const double y = lds_f64(wa);
                h0 = fma(lds_f64(qa), y, h0);
                if (nr > 33) h1 = fma(lds_f64(qa + 8u), y, h1);
                if (nr > 34) h2 = fma(lds_f64(qa + 16u), y, h2);
                qa += 32u * rs8;
                wa += 256u;
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                h0 += __shfl_xor_sync(0xffffffffu, h0, off);
                if (nr > 33) h1 += __shfl_xor_sync(0xffffffffu, h1, off);
                if (nr > 34) h2 += __shfl_xor_sync(0xffffffffu, h2, off);
            }
            hi[f] = lane == 0 ? h0 : (lane == 1 ? h1 : h2);
        }
    }
#pragma unroll
    for (int f = 0; f < FB; ++f) {
        lo[f] = (a0[f] + a1[f]) + (a2[f] + a3[f]);
#pragma unroll
        for (int off = W; off < 32; off <<= 1) lo[f] += __shfl_xor_sync(0xffffffffu, lo[f], off);
    }
}

template <int FB>
__device__ __forceinline__ void warp_matvec_fields(uint32_t op_s, uint32_t v_s, uint32_t vstride, int nfb, int n, int nr,
                                                   const Groups& gr, int lane, double (&lo)[FB], double (&hi)[FB]) {
    switch (gr.lw) {   // warp-uniform
        case 0: warp_matvec_fields_t<0, FB>(op_s, v_s, vstride, nfb, n, nr, lane, lo, hi); break;
        case 1: warp_matvec_fields_t<1, FB>(op_s, v_s, vstride, nfb, n, nr, lane, lo, hi); break;
        case 2: warp_matvec_fields_t<2, FB>(op_s, v_s, vstride, nfb, n, nr, lane, lo, hi); break;
        case 3: warp_matvec_fields_t<3, FB>(op_s, v_s, vstride, nfb, n, nr, lane, lo, hi); break;
        case 4: warp_matvec_fields_t<4, FB>(op_s, v_s, vstride, nfb, n, nr, lane, lo, hi); break;
        default: warp_matvec_fields_t<5, FB>(op_s, v_s, vstride, nfb, n, nr, lane, lo, hi); break;
    }
}

// solve_kernel for F.nf fields (ALGO_BASIC: FB fields per block of accumulators; ALGO_ITERATIVE: the fields one after
// another, each refined against the resident block with its own exit and count).  Ring and records as in solve_kernel;
// each field's fk row is one more bulk copy into its fext slot of the stage.
template <int DIM, bool ITER, bool UNI, int FB>
__global__ void __launch_bounds__(SOLVE_FIELDS_THREADS, 1) solve_fields_kernel(FieldsParams F) {
    const SolveParams& P = F.P;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int nf = F.nf;
    double* wb = reinterpret_cast<double*>(smem_raw) + (size_t)warp * P.warp_doubles;
    double* ring = wb;
    double* fis = wb + P.off_fi;
    double* rs = wb + P.off_r;
    const uint32_t rs_u32 = smem_u32(rs);
    const uint32_t fstride = (uint32_t)F.f_doubles * 8u;
    WarpRing R(smem_u32(ring), smem_u32(smem_raw + P.bar_off_bytes) + (uint32_t)(warp * P.stages) * 8u, P.stages,
               (uint32_t)P.stage_doubles * 8u, P.case_lo, P.ncases);
    const long long gw = R.first, GW = R.stride, n_my = R.n_my;

    auto get_meta = [&](long long c) { return case_meta<UNI>(P.meta, P.uni, P.op_stride, c); };
    const bool f_tma = P.f_tma != 0;
    const bool xk_tma = ITER && P.xk_tma;
    auto issue = [&](uint32_t st, uint32_t bar, long long c) {   // lane 0 only
        const CaseMeta m = get_meta(c);
        const uint32_t b_op = op_block_bytes(m);
        const uint32_t b_f = f_tma ? (((uint32_t)m.nk + 1u) & ~1u) * 8u : 0u;
        const uint32_t b_x = xk_tma ? (((uint32_t)(m.nk * DIM) + 1u) & ~1u) * 8u : 0u;
        mbar_expect_tx_u32(bar, b_op + (uint32_t)nf * b_f + b_x);
        if (b_op) tma_load_1d_u32(st, P.op + m.op_off, b_op, bar);
        if (b_f)
            for (int f = 0; f < nf; ++f)
                tma_load_1d_u32(st + (uint32_t)P.off_f * 8u + (uint32_t)f * fstride, P.fk + f * F.fk_sf + c * P.fk_s0, b_f, bar);
        if (b_x) tma_load_1d_u32(st + (uint32_t)P.off_xk * 8u, P.xk + c * P.xk_s0, b_x, bar);
    };

    R.start(lane, issue);

    int itmax = 0;
    CaseMeta mt{};
    if (n_my > 0) mt = get_meta(gw);
    long long c = gw;
    for (long long i = 0; i < n_my; ++i, c += GW) {
        R.refill(lane, i, c, issue);
        if (!UNI && R.S > 1 && lane == 0 && i + R.S < n_my) asm volatile("prefetch.global.L1 [%0];" ::"l"(P.meta + (c + (long long)R.S * GW)));
        const long long knowns = mt.knowns;
        if (UNI) mt = P.uni;
        const int nk = mt.nk, no = mt.no, nr = mt.nr, nkn = mt.nkn, nq = nk + nkn;
        double* st = ring + (size_t)R.stage * P.stage_doubles;
        const uint32_t st_u32 = R.cur();
        double* fext0 = st + P.off_f;
        const double* xks = st + P.off_xk;
        const Groups gr = make_groups(nr, lane);

        if (!f_tma) {
            for (int f = 0; f < nf; ++f) {
                const double* fp = P.fk + f * F.fk_sf + c * P.fk_s0;
                double* fx = fext0 + f * F.f_doubles;
                for (int k = lane; k < nk; k += 32) fx[k] = ld_stream(fp + (long long)k * P.fk_s1);
            }
        }
        if (ITER && !xk_tma) {
            const double* xp = P.xk + c * P.xk_s0;
            double* xw = st + P.off_xk;
            for (int t = lane; t < nk * DIM; t += 32) xw[t] = xp[(long long)(t / DIM) * P.xk_s1 + (t % DIM)];
        }
        const bool in0 = lane < no, in1 = lane + 32 < no;
        const bool unk0 = in0 && !((knowns >> lane) & 1LL);
        const bool unk1 = in1 && !((knowns >> (lane + 32)) & 1LL);
        const int below0 = __popcll(knowns & ((1LL << lane) - 1));
        const int below1 = __popcll(knowns & ((1LL << (lane + 32)) - 1));
        const int j0 = unk0 ? lane - below0 : 0;
        const int j1 = unk1 ? lane + 32 - below1 : 0;
        CaseMeta mt_next = mt;
        if (i + 1 < n_my && (!UNI || P.meta)) mt_next = get_meta(c + GW);
        __syncwarp();
        R.wait();
        // known values of every field (after the copies have landed: a copy of an odd-length row also writes fext[nk])
        if (nkn) {
            for (int f = 0; f < nf; ++f) {
                const double* fr = F.fi + f * F.fi_sf + c * F.fi_s0;
                double* fx = fext0 + f * F.f_doubles;
                if (in0 && !unk0) fx[nk + below0] = fr[lane];
                if (in1 && !unk1) fx[nk + below1] = fr[lane + 32];
            }
            __syncwarp();
        }
        const double qnan = __longlong_as_double(0x7ff8000000000000LL);

        if constexpr (!ITER) {
            if (nr > 0) {
                for (int f0 = 0; f0 < nf; f0 += FB) {
                    double lo[FB], hi[FB];
                    warp_matvec_fields<FB>(st_u32, st_u32 + (uint32_t)P.off_f * 8u + (uint32_t)f0 * fstride, fstride,
                                           min(FB, nf - f0), nq, nr, gr, lane, lo, hi);
#pragma unroll
                    for (int f = 0; f < FB; ++f) {
                        if (f0 + f >= nf) break;
                        double* fr = F.fi + (f0 + f) * F.fi_sf + c * F.fi_s0;
                        const double t0 = fetch_reduced(lo[f], hi[f], j0);
                        if (unk0) fr[lane] = nq == 0 ? qnan : t0;
                        if (no > 32) {
                            const double t1 = fetch_reduced(lo[f], hi[f], j1);
                            if (unk1) fr[lane + 32] = nq == 0 ? qnan : t1;
                        }
                    }
                }
            }
        } else {
            int itc = 0;
            for (int f = 0; f < nf; ++f) {
                const double* fext = fext0 + f * F.f_doubles;
                // known slots keep the caller's value
                double v0 = (in0 && !unk0) ? fext[nk + below0] : 0.0, v1 = (in1 && !unk1) ? fext[nk + below1] : 0.0;
                if (nr > 0) {
                    double lo, hi;
                    warp_matvec<true>(st_u32, st_u32 + (uint32_t)P.off_f * 8u + (uint32_t)f * fstride, nq, nr, gr, lane, lo, hi);
                    const double t0 = fetch_reduced(lo, hi, j0);
                    if (unk0) v0 = t0;
                    if (no > 32) {
                        const double t1 = fetch_reduced(lo, hi, j1);
                        if (unk1) v1 = t1;
                    }
                }
                if (nq == 0 && nr > 0) {
                    if (unk0) v0 = qnan;
                    if (unk1) v1 = qnan;
                }
                if (in0) fis[lane] = v0;
                if (in1) fis[lane + 32] = v1;
                __syncwarp();
                const int it = refine_case<DIM>(P, c, no, nk, nr, gr, lane, fis, xks, fext, rs, rs_u32, st_u32, unk0, unk1,
                                                j0, j1, v0, v1);
                itc = max(itc, it);
                double* fr = F.fi + f * F.fi_sf + c * F.fi_s0;
                if (unk0) fr[lane] = v0;
                if (unk1) fr[lane + 32] = v1;
                __syncwarp();   // every lane is done with fis / rs of this field
            }
            if (P.iters_case && lane == 0) P.iters_case[c] = max(P.iters_case[c], itc);
            itmax = max(itmax, itc);
        }
        R.release();
        mt = mt_next;
    }
    if (ITER && lane == 0 && itmax > 0) atomicMax(P.iters_max, itmax);
}

// solve_pack_kernel for F.nf fields: lane (cg, o) accumulates its operator column against the fk rows of FB fields at
// once (one shared-memory read of each operator element per FB fields), each field in solve_pack_kernel's order.
template <int FB>
__global__ void __launch_bounds__(SOLVE_FIELDS_THREADS) solve_pack_fields_kernel(FieldsParams F) {
    const SolveParams& P = F.P;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int nf = F.nf;
    double* ring = reinterpret_cast<double*>(smem_raw) + (size_t)warp * P.warp_doubles;
    const uint32_t fstride = (uint32_t)F.f_doubles * 8u, kstride = (uint32_t)F.k_doubles * 8u;

    const CaseMeta u = P.uni;
    const int nk = u.nk, no = u.no, nr = u.nr, nkn = u.nkn;
    const int lw = P.pack_lw, CPW = 32 >> lw;
    const int cg = lane >> lw, o = lane & ((1 << lw) - 1);
    const int ops = (int)P.op_stride;

    WarpRing R(smem_u32(ring), smem_u32(smem_raw + P.bar_off_bytes) + (uint32_t)(warp * P.stages) * 8u, P.stages,
               (uint32_t)P.stage_doubles * 8u, 0, (P.ncases - P.case_lo + CPW - 1) / CPW);   // packs, as in solve_pack_kernel

    auto pack_cases = [&](long long pk) { return (int)min((long long)CPW, P.ncases - (P.case_lo + pk * CPW)); };
    auto f_by_tma = [&](int ncs) { return P.f_tma && !((ncs * nk) & 1); };
    auto issue = [&](uint32_t st, uint32_t bar, long long pk) {   // lane 0 only
        const long long c0 = P.case_lo + pk * CPW;
        const int ncs = pack_cases(pk);
        const uint32_t b_op = (uint32_t)(ncs * ops) * 8u;
        const uint32_t b_f = f_by_tma(ncs) ? (uint32_t)(ncs * nk) * 8u : 0u;
        mbar_expect_tx_u32(bar, b_op + (uint32_t)nf * b_f);
        if (b_op) tma_load_1d_u32(st, P.op + c0 * P.op_stride, b_op, bar);
        if (b_f)
            for (int f = 0; f < nf; ++f)
                tma_load_1d_u32(st + (uint32_t)P.off_f * 8u + (uint32_t)f * fstride, P.fk + f * F.fk_sf + c0 * P.fk_s0, b_f, bar);
    };

    R.start(lane, issue);

    long long pk = R.first;
    for (long long i = 0; i < R.n_my; ++i, pk += R.stride) {
        R.refill(lane, i, pk, issue);
        const long long c0 = P.case_lo + pk * CPW;
        const int ncs = pack_cases(pk);
        const long long c = c0 + cg;
        double* st = ring + (size_t)R.stage * P.stage_doubles;
        const uint32_t st_u32 = R.cur();
        if (!f_by_tma(ncs)) {
            for (int f = 0; f < nf; ++f) {
                double* fs = st + P.off_f + f * F.f_doubles;
                const double* fp = P.fk + f * F.fk_sf;
                for (int t = lane; t < ncs * nk; t += 32) {
                    const int ci = t / nk, k = t - ci * nk;
                    fs[t] = ld_stream(fp + (c0 + ci) * P.fk_s0 + (long long)k * P.fk_s1);
                }
            }
        }
        const bool valid = cg < ncs && o < no;
        const long long knowns = (valid && P.meta) ? P.meta[c].knowns : u.knowns;
        const bool isk = (knowns >> o) & 1LL;
        const int below = __popcll(knowns & ((1LL << o) - 1));
        const int j = o - below;
        if (nkn && valid && isk)
            for (int f = 0; f < nf; ++f) st[P.off_xk + f * F.k_doubles + cg * nkn + below] = F.fi[f * F.fi_sf + c * F.fi_s0 + o];
        __syncwarp();
        R.wait();

        if (valid && !isk) {
            for (int f0 = 0; f0 < nf; f0 += FB) {
                const int nfb = min(FB, nf - f0);
                double a0[FB], a1[FB], a2[FB], a3[FB];
#pragma unroll
                for (int f = 0; f < FB; ++f) a0[f] = a1[f] = a2[f] = a3[f] = 0.0;
                const uint32_t rs8 = (uint32_t)nr * 8u;
                uint32_t pa = st_u32 + (uint32_t)(cg * ops + j) * 8u;
                uint32_t fa = st_u32 + (uint32_t)(P.off_f + cg * nk) * 8u + (uint32_t)f0 * fstride;
                int q = nk;
                for (; q >= 4; q -= 4) {
                    const double x0 = lds_f64(pa), x1 = lds_f64(pa + rs8), x2 = lds_f64(pa + 2u * rs8), x3 = lds_f64(pa + 3u * rs8);
#pragma unroll
                    for (int f = 0; f < FB; ++f) {
                        if (f < nfb) {
                            const uint32_t ff = fa + (uint32_t)f * fstride;
                            a0[f] = fma(x0, lds_f64(ff), a0[f]);
                            a1[f] = fma(x1, lds_f64(ff + 8u), a1[f]);
                            a2[f] = fma(x2, lds_f64(ff + 16u), a2[f]);
                            a3[f] = fma(x3, lds_f64(ff + 24u), a3[f]);
                        }
                    }
                    pa += 4u * rs8;
                    fa += 32u;
                }
                for (; q > 0; --q) {
                    const double x0 = lds_f64(pa);
#pragma unroll
                    for (int f = 0; f < FB; ++f)
                        if (f < nfb) a0[f] = fma(x0, lds_f64(fa + (uint32_t)f * fstride), a0[f]);
                    pa += rs8;
                    fa += 8u;
                }
                uint32_t ka = st_u32 + (uint32_t)(P.off_xk + cg * nkn) * 8u + (uint32_t)f0 * kstride;
                for (int m = 0; m < nkn; ++m) {
                    const double x0 = lds_f64(pa);
#pragma unroll
                    for (int f = 0; f < FB; ++f)
                        if (f < nfb) a1[f] = fma(x0, lds_f64(ka + (uint32_t)f * kstride), a1[f]);
                    pa += rs8;
                    ka += 8u;
                }
#pragma unroll
                for (int f = 0; f < FB; ++f) {
                    if (f >= nfb) break;
                    double v = (a0[f] + a1[f]) + (a2[f] + a3[f]);
                    if (nk + nkn == 0) v = __longlong_as_double(0x7ff8000000000000LL);
                    F.fi[(f0 + f) * F.fi_sf + c * F.fi_s0 + o] = v;
                }
            }
        }
        R.release();
    }
}

template <int DIM, bool ITER, bool UNI, int FB>
static cudaError_t launch_fields_one(const FieldsParams& F, int blocks, int threads, size_t smem, cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(solve_fields_kernel<DIM, ITER, UNI, FB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
    if (e != cudaSuccess) return e;
    solve_fields_kernel<DIM, ITER, UNI, FB><<<blocks, threads, smem, st>>>(F);
    return cudaGetLastError();
}

template <bool UNI>
static cudaError_t launch_fields_basic(const FieldsParams& F, int blocks, int threads, size_t smem, cudaStream_t st) {
    if (F.nf <= 1) return launch_fields_one<1, false, UNI, 1>(F, blocks, threads, smem, st);
    if (F.nf <= 2) return launch_fields_one<1, false, UNI, 2>(F, blocks, threads, smem, st);
    if (F.nf <= 4) return launch_fields_one<1, false, UNI, 4>(F, blocks, threads, smem, st);
    return launch_fields_one<1, false, UNI, SOLVE_FIELDS_BLOCK>(F, blocks, threads, smem, st);
}

cudaError_t launch_solve_fields(int dim, const FieldsParams& F, int blocks, int threads, size_t smem, cudaStream_t st) {
    const bool uni = F.P.meta == nullptr || F.P.geom_uniform;
    if (F.P.algorithm != WLSQM_ALGO_ITERATIVE)
        return uni ? launch_fields_basic<true>(F, blocks, threads, smem, st) : launch_fields_basic<false>(F, blocks, threads, smem, st);
    if (dim == 1) return uni ? launch_fields_one<1, true, true, 1>(F, blocks, threads, smem, st)
                             : launch_fields_one<1, true, false, 1>(F, blocks, threads, smem, st);
    if (dim == 2) return uni ? launch_fields_one<2, true, true, 1>(F, blocks, threads, smem, st)
                             : launch_fields_one<2, true, false, 1>(F, blocks, threads, smem, st);
    return uni ? launch_fields_one<3, true, true, 1>(F, blocks, threads, smem, st)
               : launch_fields_one<3, true, false, 1>(F, blocks, threads, smem, st);
}

template <int FB>
static cudaError_t launch_pack_fields_one(const FieldsParams& F, int blocks, int threads, size_t smem, cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(solve_pack_fields_kernel<FB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    solve_pack_fields_kernel<FB><<<blocks, threads, smem, st>>>(F);
    return cudaGetLastError();
}

cudaError_t launch_solve_pack_fields(const FieldsParams& F, int blocks, int threads, size_t smem, cudaStream_t st) {
    if (F.nf <= 1) return launch_pack_fields_one<1>(F, blocks, threads, smem, st);
    if (F.nf <= 2) return launch_pack_fields_one<2>(F, blocks, threads, smem, st);
    if (F.nf <= 4) return launch_pack_fields_one<4>(F, blocks, threads, smem, st);
    return launch_pack_fields_one<SOLVE_FIELDS_BLOCK>(F, blocks, threads, smem, st);
}

}  // namespace wlsqm
