// wlsqm_solve.cu -- K2: the per-time-step solve as ONE streaming pass over the stored operators.
//
// Replaces ExpertSolver.solve's per-case work (wlsqm/fitter/expert.pyx:467-655):
//   Case_set_fi / Case_get_fi   wlsqm/fitter/infra.pyx:780-795
//   impl.solve / solve_contig   wlsqm/fitter/impl.pyx:731-846 / 861-974   (RHS, knowns elimination, dgetrs, sens)
//   impl.solve_iterative        wlsqm/fitter/impl.pyx:986-1083             (data-space refinement)
//
// Layout / dataflow.  prepare() left, for every case, one contiguous block Op[(nk+nkn)][nr] in HBM
// (wlsqm_prepare.cu).  Each warp owns a ring of shared-memory stages; one elected lane streams the
// next cases' blocks into the ring with 1D bulk TMA (cp.async.bulk + mbarrier complete_tx) while
// the warp works on the current one, so HBM sees long, fully used, 16 B-aligned bursts and no
// register is spent on loads in flight.  With the block resident in shared memory:
//   fi[r2o[j]]  = sum_q Op[q][j] * fext[q],   fext = (fk[0..nk), known fi values)
//   sens[k][o]  = Op[k][j(o)]  (NaN for known o)                      -- no extra solves
//   ALGO_ITERATIVE: r_k = fk_k - model(xk_k); stop if max|r| == previous max|r| exactly
//                   (impl.pyx:1057-1060); fi[unknown] += Op[:nk]^T r    -- operator is not re-read from HBM
// Results go to the solver-owned fi copy (the reference's Case.fi, read later by interpolate) and,
// when the caller's fi is device memory that cannot alias fk, straight to it as well; otherwise the
// deferred write-back of expert.pyx:548-557 is a second tiny kernel (scatter_fi_kernel).
#include <type_traits>
#include "wlsqm_common.cuh"
#include "wlsqm_kernels.h"
#include "wlsqm_solve_common.cuh"

namespace wlsqm {

// UNI = the whole batch shares one CaseMeta (passed by value): everything derived from it is loop
// invariant and hoisted by the compiler, which is what keeps the per-case instruction count low.
template <int DIM, bool ITER, bool SENS, bool UNI>
__global__ void __launch_bounds__(ITER ? (DIM == 3 ? SOLVE_MAX_THREADS_ITER : SOLVE_ITER12_THREADS) : SOLVE_MAX_THREADS, 1)
solve_kernel(SolveParams P) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    double* wb = reinterpret_cast<double*>(smem_raw) + (size_t)warp * P.warp_doubles;
    double* ring = wb;                      // S stages of [operator block | fext = (fk, known fi) | xk (ITER)]
    double* fis = wb + P.off_fi;            // current solution of the case (no values)
    double* rs = wb + P.off_r;              // ITER: residual at the neighbours
    const uint32_t rs_u32 = smem_u32(rs);
    WarpRing R(smem_u32(ring), smem_u32(smem_raw + P.bar_off_bytes) + (uint32_t)(warp * P.stages) * 8u, P.stages,
               (uint32_t)P.stage_doubles * 8u, P.case_lo, P.ncases);
    const long long gw = R.first, GW = R.stride, n_my = R.n_my;

    auto get_meta = [&](long long c) { return case_meta<UNI>(P.meta, P.uni, P.op_stride, c); };
    // bulk copies need 16 B alignment and sizes: the host says whether the arrays qualify (f_tma, xk_tma: 16 B aligned
    // base, unit stride, EVEN row pitch); otherwise the lanes gather with plain loads.  A row with an odd element count is
    // copied with one element more -- the pitch is even, so that element exists, and nothing reads it (fext[nk] is either
    // unused or the first known value, which the lanes then store AFTER the copy has landed: `late_knowns` below).  A lane
    // gather instead would put an unprefetched global load on the critical path of every such case.
    auto f_by_tma = [&](const CaseMeta&) { return P.f_tma != 0; };
    auto xk_by_tma = [&](const CaseMeta&) { return ITER && P.xk_tma; };
    auto issue = [&](uint32_t st, uint32_t bar, long long c) {   // lane 0 only: arm the stage's barrier and start its copies
        const CaseMeta m = get_meta(c);
        const uint32_t b_op = op_block_bytes(m);
        const uint32_t b_f = f_by_tma(m) ? (((uint32_t)m.nk + 1u) & ~1u) * 8u : 0u;
        const uint32_t b_x = xk_by_tma(m) ? (((uint32_t)(m.nk * DIM) + 1u) & ~1u) * 8u : 0u;
        mbar_expect_tx_u32(bar, b_op + b_f + b_x);
        if (b_op) tma_load_1d_u32(st, P.op + m.op_off, b_op, bar);
        if (b_f) tma_load_1d_u32(st + (uint32_t)P.off_f * 8u, P.fk + c * P.fk_s0, b_f, bar);
        if (b_x) tma_load_1d_u32(st + (uint32_t)P.off_xk * 8u, P.xk + c * P.xk_s0, b_x, bar);
    };
    // known fi values of a case, one register per lane and 32-slot group (prefetched one case ahead)
    auto load_g = [&](long long c, const CaseMeta& m, double& g0, double& g1) {
        g0 = g1 = 0.0;
        if (lane < m.no && ((m.knowns >> lane) & 1LL)) g0 = P.fi_in[c * P.fi_in_s0 + lane];
        if (lane + 32 < m.no && ((m.knowns >> (lane + 32)) & 1LL)) g1 = P.fi_in[c * P.fi_in_s0 + lane + 32];
    };

    R.start(lane, issue);

    int itmax = 0;
    double g0 = 0.0, g1 = 0.0;
    CaseMeta mt{};
    if (n_my > 0) {
        mt = get_meta(gw);
        if (mt.nkn) load_g(gw, mt, g0, g1);
    }
    long long c = gw;
    for (long long i = 0; i < n_my; ++i, c += GW) {
        R.refill(lane, i, c, issue);
        // per-case records: the one lane 0 needs at the top of the NEXT iteration (to start the copies of the case after
        // next) is requested into L1 now -- fetched cold it held up the whole warp there (17 % of the stall samples of the
        // mixed-size kernel, profiles/r02_solve_kernel_hetero_source_lines.txt)
        // (with a one-stage ring the record in question is the next case's, which every lane fetches below anyway)
        if (!UNI && R.S > 1 && lane == 0 && i + R.S < n_my) asm volatile("prefetch.global.L1 [%0];" ::"l"(P.meta + (c + (long long)R.S * GW)));
        const long long knowns = mt.knowns;
        if (UNI) mt = P.uni;   // loop invariant: lets the compiler hoist everything derived from the record
        const int nk = mt.nk, no = mt.no, nr = mt.nr, nkn = mt.nkn, nq = nk + nkn;
        double* st = ring + (size_t)R.stage * P.stage_doubles;
        const uint32_t st_u32 = R.cur();
        const double* op = st;
        double* fext = st + P.off_f;
        const double* xks = st + P.off_xk;
        const Groups gr = make_groups(nr, lane);

        // ---- data that did not come by TMA, and the known values ---------------------------------
        if (!f_by_tma(mt)) {
            const double* f = P.fk + c * P.fk_s0;
            for (int k = lane; k < nk; k += 32) fext[k] = ld_stream(f + (long long)k * P.fk_s1);
        }
        if (ITER && !xk_by_tma(mt)) {
            const double* xp = P.xk + c * P.xk_s0;
            double* xw = st + P.off_xk;
            for (int t = lane; t < nk * DIM; t += 32) xw[t] = xp[(long long)(t / DIM) * P.xk_s1 + (t % DIM)];
        }
        // reduced index of the slots this lane writes back: o = lane and o = lane + 32
        const bool in0 = lane < no, in1 = lane + 32 < no;
        const bool unk0 = in0 && !((knowns >> lane) & 1LL);
        const bool unk1 = in1 && !((knowns >> (lane + 32)) & 1LL);
        const int below0 = __popcll(knowns & ((1LL << lane) - 1));
        const int below1 = __popcll(knowns & ((1LL << (lane + 32)) - 1));
        const int j0 = unk0 ? lane - below0 : 0;
        const int j1 = unk1 ? lane + 32 - below1 : 0;
        const bool late_knowns = f_by_tma(mt) && (nk & 1);      // (warp-uniform) the copy writes fext[nk] too
        if (nkn && !late_knowns) {
            if (in0 && !unk0) fext[nk + below0] = g0;
            if (in1 && !unk1) fext[nk + below1] = g1;
        }
        // prefetch the next case's record and known values while this one is being worked on
        CaseMeta mt_next = mt;
        double gn0 = 0.0, gn1 = 0.0;
        if (i + 1 < n_my) {
            if (!UNI || P.meta) mt_next = get_meta(c + GW);
            if (mt_next.nkn) load_g(c + GW, mt_next, gn0, gn1);
        }
        __syncwarp();
        R.wait();
        if (nkn && late_knowns) {
            if (in0 && !unk0) fext[nk + below0] = g0;
            if (in1 && !unk1) fext[nk + below1] = g1;
            __syncwarp();
        }

        // ---- fi[unknown] = Op^T fext ----------------------------------------------------------------
        double v0 = g0, v1 = g1;     // known slots keep the caller's value
        if (nr > 0) {
            double lo, hi;
            warp_matvec<ITER>(st_u32, st_u32 + (uint32_t)P.off_f * 8u, nq, nr, gr, lane, lo, hi);
            const double t0 = fetch_reduced(lo, hi, j0);
            if (unk0) v0 = t0;
            if (no > 32) {
                const double t1 = fetch_reduced(lo, hi, j1);
                if (unk1) v1 = t1;
            }
        }
        if (nq == 0 && nr > 0) {
            // no neighbours and nothing known: the reference factors an all-zero matrix and returns NaN
            if (unk0) v0 = __longlong_as_double(0x7ff8000000000000LL);
            if (unk1) v1 = __longlong_as_double(0x7ff8000000000000LL);
        }
        if (ITER) {
            if (in0) fis[lane] = v0;
            if (in1) fis[lane + 32] = v1;
            __syncwarp();
        }

        // ---- sensitivities: the operator itself, re-indexed by DOF slot (impl.pyx:838-846) ------
        if (SENS && nr > 0) {   // nr == 0: silent no-op, sens untouched (impl.pyx:742)
            double* sn = P.sens + c * P.sens_s0;
            const double qnan = __longlong_as_double(0x7ff8000000000000LL);
            if (no <= 32) {
                // the 32 lanes cover G2 = 32 / W2 operator rows per pass (W2 = smallest power of two >= no);
                // a lane's DOF slot, its reduced index and its NaN flag do not change from pass to pass
                const int lw2 = no <= 1 ? 0 : 32 - __clz(no - 1);
                const int G2 = 32 >> lw2, rg = lane >> lw2, o = lane & ((1 << lw2) - 1);
                const bool kn = (knowns >> o) & 1LL;
                const int jo = o - __popcll(knowns & ((1LL << o) - 1));
                if (o < no) {
                    double* sp = sn + (long long)rg * P.sens_s1 + o;
                    const double* opp = op + rg * nr + jo;
                    const long long dsn = (long long)G2 * P.sens_s1;
                    const int dop = G2 * nr;
                    for (int k = rg; k < nk; k += G2) {
                        st_stream(sp, kn ? qnan : *opp);
                        sp += dsn;
                        opp += dop;
                    }
                }
            } else {
                // columns 0..31 of every row: one store per row; columns 32..no-1 (at most three): the 32 lanes take
                // the tails of TR = 32 / nt rows per store instead of one nearly empty store per row
                double* sp = sn + lane;
                const double* opp = op;
#pragma unroll 4
                for (int k = 0; k < nk; ++k) {
                    st_stream(sp, unk0 ? opp[j0] : qnan);
                    sp += P.sens_s1;
                    opp += nr;
                }
                const int nt = no - 32, TR = 32 / nt;
                const int tr = lane / nt, to = 32 + lane % nt;
                if (tr < TR) {
                    const bool tkn = (knowns >> to) & 1LL;
                    const int tj = to - __popcll(knowns & ((1LL << to) - 1));
                    for (int k = tr; k < nk; k += TR)
                        st_stream(sn + (long long)k * P.sens_s1 + to, tkn ? qnan : op[k * nr + tj]);
                }
            }
        }

        // ---- ALGO_ITERATIVE: refinement against the data (impl.pyx:1010-1083) --------------------
        if (ITER) {
            const int it = refine_case<DIM>(P, c, no, nk, nr, gr, lane, fis, xks, fext, rs, rs_u32, st_u32, unk0, unk1, j0, j1,
                                            v0, v1);
            if (P.iters_case && lane == 0) P.iters_case[c] = it;
            itmax = max(itmax, it);
        }

        // ---- write-back: solver-owned copy (all `no` entries) and, if allowed, the caller's fi ---
        if (in0) {
            if (P.fi_case) P.fi_case[c * P.fi_case_ld + lane] = v0;
            if (P.fi_out && unk0) P.fi_out[c * P.fi_out_s0 + lane] = v0;
        }
        if (in1) {
            if (P.fi_case) P.fi_case[c * P.fi_case_ld + lane + 32] = v1;
            if (P.fi_out && unk1) P.fi_out[c * P.fi_out_s0 + lane + 32] = v1;
        }
        if (P.ngather) {
            // fused all-gather: the whole row (knowns included) into every GPU's copy of the global array (peer stores
            // over NVLink; 8 * no bytes per peer against the 8 * nq * nr bytes of the block just streamed)
            const long long g = (P.gather_row0 + c) * P.gather_s0;
#pragma unroll 1
            // (rows padded to whole 128 B lines: the padding lanes store zeros, so that every row crosses NVLink as full-line
            // writes instead of two partial ones with byte enables)
            const bool w0 = in0 || (P.gather_full && lane < (int)P.gather_s0);
            const double s0v = in0 ? v0 : 0.0;
            for (int p = 0; p < P.ngather; ++p) {
                if (w0) P.gather[p][g + lane] = s0v;
                if (in1) P.gather[p][g + lane + 32] = v1;
            }
        }
        R.release();
        mt = mt_next; g0 = gn0; g1 = gn1;
    }
    if (ITER && lane == 0 && itmax > 0) atomicMax(P.iters_max, itmax);
}

// ---------------------------------------------------------------------------------------------------------
// Packed variant for small models (no <= 16, ALGO_BASIC, every case with the same sizes): a warp takes
// CPW = 32 / W consecutive cases per pass (W = smallest power of two >= no), so that the per-pass work
// -- one bulk copy of CPW contiguous operator blocks, one of CPW fk rows, barrier wait, write-back -- is shared
// by CPW cases.  Lane (cg, o) owns DOF slot o of case cg: an unknown slot accumulates its whole operator
// column over q (four independent FMA chains, no cross-lane reduction), a known slot passes its value on.
// Same arithmetic as solve_kernel; only the summation order over q differs (sequential per column).
template <bool SENS>
__global__ void __launch_bounds__(SOLVE_MAX_THREADS) solve_pack_kernel(SolveParams P) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    double* ring = reinterpret_cast<double*>(smem_raw) + (size_t)warp * P.warp_doubles;

    const CaseMeta u = P.uni;
    const int nk = u.nk, no = u.no, nr = u.nr, nkn = u.nkn;
    const int lw = P.pack_lw, CPW = 32 >> lw;
    const int cg = lane >> lw, o = lane & ((1 << lw) - 1);
    const int ops = (int)P.op_stride;                         // doubles per operator block (even)

    // units are packs, counted from 0: pack pk holds the cases from case_lo + pk * CPW on
    WarpRing R(smem_u32(ring), smem_u32(smem_raw + P.bar_off_bytes) + (uint32_t)(warp * P.stages) * 8u, P.stages,
               (uint32_t)P.stage_doubles * 8u, 0, (P.ncases - P.case_lo + CPW - 1) / CPW);
    const long long gw = R.first, GW = R.stride, n_my = R.n_my;

    auto pack_cases = [&](long long pk) { return (int)min((long long)CPW, P.ncases - (P.case_lo + pk * CPW)); };
    auto f_by_tma = [&](int ncs) { return P.f_tma && !((ncs * nk) & 1); };
    auto issue = [&](uint32_t st, uint32_t bar, long long pk) {   // lane 0 only
        const long long c0 = P.case_lo + pk * CPW;
        const int ncs = pack_cases(pk);
        const uint32_t b_op = (uint32_t)(ncs * ops) * 8u;
        const uint32_t b_f = f_by_tma(ncs) ? (uint32_t)(ncs * nk) * 8u : 0u;
        mbar_expect_tx_u32(bar, b_op + b_f);
        if (b_op) tma_load_1d_u32(st, P.op + c0 * P.op_stride, b_op, bar);
        if (b_f) tma_load_1d_u32(st + (uint32_t)P.off_f * 8u, P.fk + c0 * P.fk_s0, b_f, bar);
    };
    // knowns pattern and known value of this lane's slot in pack pk
    auto load_slot = [&](long long pk, long long& kn, double& g) {
        const long long c = P.case_lo + pk * CPW + cg;
        kn = u.knowns;
        g = 0.0;
        if (c < P.ncases && o < no) {
            if (P.meta) kn = P.meta[c].knowns;
            if ((kn >> o) & 1LL) g = P.fi_in[c * P.fi_in_s0 + o];
        }
    };

    R.start(lane, issue);

    long long knowns = u.knowns;
    double g = 0.0;
    if (n_my > 0 && (nkn || P.meta)) load_slot(gw, knowns, g);
    long long pk = gw;
    for (long long i = 0; i < n_my; ++i, pk += GW) {
        R.refill(lane, i, pk, issue);
        const long long c0 = P.case_lo + pk * CPW;
        const int ncs = pack_cases(pk);
        const long long c = c0 + cg;
        double* st = ring + (size_t)R.stage * P.stage_doubles;
        const uint32_t st_u32 = R.cur();
        double* fs = st + P.off_f;                 // [CPW][nk]   fk rows of the pack
        double* ks = st + P.off_xk;                // [CPW][nkn]  known values of the pack
        if (!f_by_tma(ncs)) {
            for (int t = lane; t < ncs * nk; t += 32) {
                const int ci = t / nk, k = t - ci * nk;
                fs[t] = ld_stream(P.fk + (c0 + ci) * P.fk_s0 + (long long)k * P.fk_s1);
            }
        }
        const bool valid = cg < ncs && o < no;
        const bool isk = (knowns >> o) & 1LL;
        const int below = __popcll(knowns & ((1LL << o) - 1));
        const int j = o - below;
        if (nkn && valid && isk) ks[cg * nkn + below] = g;
        // the next pack's knowns pattern and known values travel while this one is being worked on
        long long kn_next = u.knowns;
        double g_next = 0.0;
        if (i + 1 < n_my && (nkn || P.meta)) load_slot(pk + GW, kn_next, g_next);
        __syncwarp();
        R.wait();

        // ---- fi[unknown slot] = its operator column . fext ------------------------------------------------
        double v = g;
        if (valid && !isk) {
            double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
            const uint32_t rs8 = (uint32_t)nr * 8u;
            uint32_t pa = st_u32 + (uint32_t)(cg * ops + j) * 8u;
            uint32_t fa = st_u32 + (uint32_t)(P.off_f + cg * nk) * 8u;
            int q = nk;
            for (; q >= 4; q -= 4) {
                const double x0 = lds_f64(pa), x1 = lds_f64(pa + rs8), x2 = lds_f64(pa + 2u * rs8), x3 = lds_f64(pa + 3u * rs8);
                const double y0 = lds_f64(fa), y1 = lds_f64(fa + 8u), y2 = lds_f64(fa + 16u), y3 = lds_f64(fa + 24u);
                a0 = fma(x0, y0, a0);
                a1 = fma(x1, y1, a1);
                a2 = fma(x2, y2, a2);
                a3 = fma(x3, y3, a3);
                pa += 4u * rs8;
                fa += 32u;
            }
            for (; q > 0; --q) {
                a0 = fma(lds_f64(pa), lds_f64(fa), a0);
                pa += rs8;
                fa += 8u;
            }
            uint32_t ka = st_u32 + (uint32_t)(P.off_xk + cg * nkn) * 8u;
            for (int m = 0; m < nkn; ++m) {
                a1 = fma(lds_f64(pa), lds_f64(ka), a1);
                pa += rs8;
                ka += 8u;
            }
            v = (a0 + a1) + (a2 + a3);
            // no neighbours and nothing known: the reference factors an all-zero matrix and returns NaN
            if (nk + nkn == 0) v = __longlong_as_double(0x7ff8000000000000LL);
        }
        if (valid) {
            if (P.fi_case) P.fi_case[c * P.fi_case_ld + o] = v;
            if (P.fi_out && !isk) P.fi_out[c * P.fi_out_s0 + o] = v;
            if (P.ngather) {
                const long long g = (P.gather_row0 + c) * P.gather_s0 + o;
#pragma unroll 1
                for (int p = 0; p < P.ngather; ++p) P.gather[p][g] = v;
            }
        }
        // ---- sensitivities: the operator itself, re-indexed by DOF slot (impl.pyx:838-846) ----------------
        if (SENS && nr > 0) {
            const double qnan = __longlong_as_double(0x7ff8000000000000LL);
            if (valid) {
                double* sp = P.sens + c * P.sens_s0 + o;
                const double* opp = st + cg * ops + j;
                for (int k = 0; k < nk; ++k) {
                    st_stream(sp, isk ? qnan : *opp);
                    sp += P.sens_s1;
                    opp += nr;
                }
            }
        }
        R.release();
        knowns = kn_next;
        g = g_next;
    }
}

cudaError_t launch_solve_pack(const SolveParams& P, int blocks, int threads, size_t smem, cudaStream_t st) {
    cudaError_t e;
    if (P.sens) {
        e = cudaFuncSetAttribute(solve_pack_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        solve_pack_kernel<true><<<blocks, threads, smem, st>>>(P);
    } else {
        e = cudaFuncSetAttribute(solve_pack_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        solve_pack_kernel<false><<<blocks, threads, smem, st>>>(P);
    }
    return cudaGetLastError();
}

// Deferred write-back (expert.pyx:548-557): caller's fi <- solver-owned copy, first no_j columns.
__global__ void scatter_fi_kernel(const CaseMeta* meta, CaseMeta uni, long long ncases, const double* fi_case,
                                  int ld, double* fi_out, long long s0) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long c = t / ld;
    const int o = (int)(t - c * ld);
    if (c >= ncases) return;
    const int no = meta ? meta[c].no : uni.no;
    if (o < no) fi_out[c * s0 + o] = fi_case[c * ld + o];
}

template <int DIM, bool ITER, bool SENS, bool UNI>
static cudaError_t launch_one(const SolveParams& P, int blocks, int threads, size_t smem, cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(solve_kernel<DIM, ITER, SENS, UNI>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
    if (e != cudaSuccess) return e;
    solve_kernel<DIM, ITER, SENS, UNI><<<blocks, threads, smem, st>>>(P);
    return cudaGetLastError();
}

template <int DIM, bool ITER>
static cudaError_t launch_su(const SolveParams& P, int blocks, int threads, size_t smem, cudaStream_t st) {
    const bool sens = P.sens != nullptr, uni = P.meta == nullptr || P.geom_uniform;
    if (sens) return uni ? launch_one<DIM, ITER, true, true>(P, blocks, threads, smem, st)
                         : launch_one<DIM, ITER, true, false>(P, blocks, threads, smem, st);
    return uni ? launch_one<DIM, ITER, false, true>(P, blocks, threads, smem, st)
               : launch_one<DIM, ITER, false, false>(P, blocks, threads, smem, st);
}

cudaError_t launch_solve(int dim, const SolveParams& P, int blocks, int threads, size_t smem, cudaStream_t st) {
    if (P.algorithm != WLSQM_ALGO_ITERATIVE) return launch_su<1, false>(P, blocks, threads, smem, st);
    if (dim == 1) return launch_su<1, true>(P, blocks, threads, smem, st);
    if (dim == 2) return launch_su<2, true>(P, blocks, threads, smem, st);
    return launch_su<3, true>(P, blocks, threads, smem, st);
}

cudaError_t launch_scatter_fi(const CaseMeta* meta, const CaseMeta& uni, long long ncases, const double* fi_case,
                              int fi_case_ld, double* fi_out, long long fi_out_s0, cudaStream_t st) {
    const long long total = ncases * fi_case_ld;
    if (total == 0) return cudaSuccess;
    const int threads = 256;
    const long long blocks = (total + threads - 1) / threads;
    scatter_fi_kernel<<<(unsigned)blocks, threads, 0, st>>>(meta, uni, ncases, fi_case, fi_case_ld, fi_out, fi_out_s0);
    return cudaGetLastError();
}

}  // namespace wlsqm
