// wlsqm_operator.cu -- export of the prepared solution operators: per-case stencil weights and a global CSR matrix.
//
// The exported quantity is the reference's `sens` (wlsqm/fitter/impl.pyx:769-779, d fi / d fk), which callers of
// the reference turn into Jacobians of implicit steps, here contracted with caller-given coefficient rows and
// assembled over the point cloud of prepare_hoods() without ever forming the dense (ncases, nk, no) array.
//
// Definitions (DESIGN.md §4 K6).  prepare() left, per case, Op[q][j] (q < nk: d fi[r2o[j]] / d fk[q]; q = nk + t:
// d fi[r2o[j]] / d fi[t-th known slot]).  For a coefficient row c (one operator) and case i:
//   W[i][k] = sum_{unknown s < no, c[s] != 0, ascending s} c[s] * Op[k][j(s)]            (FMA chain from 0), k < nk
//   K[i][m] = (the same sum over Op[nk + t(m)][j(s)]) + c[m]                             known m < no
// Zero coefficients are skipped, never multiplied: a NaN entry of a block reaches only the operators that use it.
// CSR row i holds, per distinct neighbour index p, the W[i][k] with hoods[i][k] == p summed in ascending k; with
// centre folding, the known-F weight K[i][0] is added last to column center + i and reported as 0 in K.
//
// stencil_kernel: one warp per case streams its block through the shared-memory ring of solve_kernel (WarpRing, same
// CaseMeta addressing, case_meta / op_block_bytes in wlsqm_kernels.h) and produces all nops
// operators from that one read; the coefficients live in shared memory.  Bound by the HBM read of the blocks.
// csr_kernel<false>: distinct columns per row (count); cub exclusive scan; csr_kernel<true>: columns in ascending
// order, merged values (fill).  A warp per row; the row's used hood indices are staged in shared memory.
//
// Interpolation operators (include/wlsqm_b200.h, DESIGN.md §4 K6): the rows at query points q with model I[q] are the
// node rows of that model contracted with c_q = (Taylor terms at x[q] - xi[I[q]]) applied to the coefficients.  The
// queries are sorted stably by I (cub radix sort of 32-bit keys, run-length encoding, scan); interp_stencil_kernel
// takes one run per warp, streams the model's block once through the ring of stencil_kernel and writes each query's
// rows at the query's own position through the same contract_case.  csr_kernel<., ., true> maps row q to case I[q].
//
// Continuous mode (DESIGN.md §4 K6c): the rows are the (query, model) pairs of the models within r (the ball search over
// the model grid), each the nearest-mode row scaled by the pair's normalised weight (cont_weights_kernel,
// interp_stencil_kernel<., true>).  A query's CSR row merges its pairs' candidates: one warp sorts a short row in shared
// memory (cont_row_kernel); longer rows take a stable segmented sort over chunks of queries.
#include <cub/cub.cuh>
#include "wlsqm_common.cuh"
#include "wlsqm_kernels.h"

namespace wlsqm {

constexpr int OPX_MAX_THREADS = 1024;
constexpr int CSR_MAX_WARPS = 8;

// sum over the unknown slots with a nonzero coefficient, ascending, of c[s] * row[j(s)] (FMA chain from 0)
__device__ __forceinline__ double contract(const double* co, unsigned long long bits, unsigned long long knowns, const double* row) {
    double acc = 0.0;
    for (; bits; bits &= bits - 1) {
        const int s = __ffsll((long long)bits) - 1;
        const int j = s - __popcll(knowns & ((1ull << s) - 1));
        acc = fma(co[s], row[j], acc);
    }
    return acc;
}

// The rows of one case (one warp) for nops coefficient rows cs (stride maxno, nonzero slots nzm): W[o][row][k] (lane = k),
// K[o][row][s] and the known-F weight kf[o][row] (lane = known slot s, its row of the block is nk + its position among
// the knowns).  Operator o of W / K / kf lies o * nrows rows after the pointer given.  stencil_kernel and
// interp_stencil_kernel both write their rows here, so that the two definitions cannot drift apart.
__device__ __forceinline__ void contract_case(const double* op, const CaseMeta& m, const double* cs, const unsigned long long* nzm,
                                              int nops, int maxno, int maxnk, long long nrows, long long row, double* W,
                                              double* K, double* kf, int lane) {
    const int nk = m.nk, no = m.no, nr = m.nr;
    const unsigned long long knowns = (unsigned long long)m.knowns;
    const unsigned long long unk = ~knowns & ((1ull << no) - 1);     // no <= 35
    for (int k = lane; k < maxnk; k += 32) {
        const double* r = op + k * nr;
        double* w = W + row * maxnk + k;
        for (int o = 0; o < nops; ++o) {
            const double v = k < nk ? contract(cs + o * maxno, nzm[o] & unk, knowns, r) : 0.0;
            w[(long long)o * nrows * maxnk] = v;
        }
    }
    if (K || kf) {
        for (int s = lane; s < maxno; s += 32) {
            const bool kn = s < no && ((knowns >> s) & 1ull);
            const double* r = op + (nk + __popcll(knowns & ((1ull << s) - 1))) * nr;
            for (int o = 0; o < nops; ++o) {
                double v = 0.0;
                if (kn) v = contract(cs + o * maxno, nzm[o] & unk, knowns, r) + cs[o * maxno + s];
                if (kf && s == 0) {
                    kf[(long long)o * nrows + row] = v;   // folded into the fold column of the CSR row
                    v = 0.0;
                }
                if (K) K[((long long)o * nrows + row) * maxno + s] = v;
            }
        }
    }
}

// bit s set: coefficient s of the row co (maxno entries) is nonzero (every lane of the warp calls it)
__device__ __forceinline__ unsigned long long nonzero_slots(const double* co, int maxno, int lane) {
    const unsigned lo = __ballot_sync(0xffffffffu, lane < maxno && co[lane] != 0.0);
    const unsigned hi = __ballot_sync(0xffffffffu, lane + 32 < maxno && co[lane + 32] != 0.0);
    return ((unsigned long long)hi << 32) | lo;
}

// The CTA's copy of the coefficient rows cs [nops][maxno] and their nonzero slots nzm [nops] (every thread calls it;
// shared memory the CTA wrote before the call is visible after it)
__device__ __forceinline__ void stage_coefficients(const double* coef, int nops, int maxno, double* cs, unsigned long long* nzm) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    for (int t = threadIdx.x; t < nops * maxno; t += blockDim.x) cs[t] = coef[t];
    __syncthreads();
    for (int o = warp; o < nops; o += nwarps) {
        const unsigned long long nz = nonzero_slots(cs + o * maxno, maxno, lane);
        if (lane == 0) nzm[o] = nz;
    }
    __syncthreads();
}

template <bool UNI>
__global__ void __launch_bounds__(OPX_MAX_THREADS, 1) stencil_kernel(StencilParams P) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int nops = P.nops, maxno = P.maxno;
    double* cs = reinterpret_cast<double*>(smem_raw);                                      // [nops][maxno]
    unsigned long long* nzm = reinterpret_cast<unsigned long long*>(cs + nops * maxno);     // [nops] nonzero slots
    stage_coefficients(P.coef, nops, maxno, cs, nzm);

    const double* ring = reinterpret_cast<double*>(smem_raw) + P.ring_off + (size_t)warp * P.stages * P.stage_doubles;
    WarpRing R(smem_u32(ring), smem_u32(smem_raw + P.bar_off_bytes) + (uint32_t)(warp * P.stages) * 8u, P.stages,
               (uint32_t)P.stage_doubles * 8u, 0, P.ncases);
    auto issue = [&](uint32_t st, uint32_t bar, long long c) {   // lane 0 only
        const CaseMeta m = case_meta<UNI>(P.meta, P.uni, P.op_stride, c);
        const uint32_t b = op_block_bytes(m);
        mbar_expect_tx_u32(bar, b);
        if (b) tma_load_1d_u32(st, P.op + m.op_off, b, bar);
    };
    R.start(lane, issue);

    long long c = R.first;
    for (long long i = 0; i < R.n_my; ++i, c += R.stride) {
        R.refill(lane, i, c, issue);
        const CaseMeta m = case_meta<UNI>(P.meta, P.uni, P.op_stride, c);
        const double* op = ring + (size_t)R.stage * P.stage_doubles;
        R.wait();
        contract_case(op, m, cs, nzm, nops, maxno, P.maxnk, P.ncases, c, P.W, P.K, P.kf, lane);
        R.release();
    }
}

cudaError_t launch_stencils(const StencilParams& P, int blocks, int threads, size_t smem, cudaStream_t st) {
    const bool uni = P.meta == nullptr || P.geom_uniform;
    cudaError_t e;
    if (uni) {
        e = cudaFuncSetAttribute(stencil_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        stencil_kernel<true><<<blocks, threads, smem, st>>>(P);
    } else {
        e = cudaFuncSetAttribute(stencil_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        stencil_kernel<false><<<blocks, threads, smem, st>>>(P);
    }
    return cudaGetLastError();
}

// ---- interpolation operators -----------------------------------------------------------------------------------
// slot exponents (a | b << 4 | c << 8) per dimension, for runtime slot indices
struct SlotExpTable { unsigned short e[3][WLSQM_MAXNO]; };
constexpr SlotExpTable make_slot_exp_table() {
    SlotExpTable t{};
    for (int s = 0; s < WLSQM_MAXNO; ++s) {
        const SlotExp e1 = slot_exp_1d(s), e2 = slot_exp_2d(s), e3 = slot_exp_3d(s);
        t.e[0][s] = (unsigned short)(e1.a | (e1.b << 4) | (e1.c << 8));
        t.e[1][s] = (unsigned short)(e2.a | (e2.b << 4) | (e2.c << 8));
        t.e[2][s] = (unsigned short)(e3.a | (e3.b << 4) | (e3.c << 8));
    }
    return t;
}
__constant__ SlotExpTable c_slot_exp = make_slot_exp_table();

// One warp per run of queries with the same case m: the case's block is streamed once (the ring of stencil_kernel),
// then for each query q of the run the lanes form the coefficient rows
//   c_q[o][s] = sum_{D ascending, coef[o][D] != 0} coef[o][D] * T_D(s),  T_D(s) = (tx[a-p] * ty[b-r]) * tz[c-u]
// (each product and sum rounded on its own: __dmul_rn / __dadd_rn cannot be contracted), with t[n] = t[n-1] * st[n-1]
// the Taylor terms of the offset h = x[q] - xi[m] per axis (st = steps_of(h)), and contract them with the block
// (contract_case) into row q.  A term with T_D(s) = 0 is not added: the sum starts at +0 and never becomes -0, so
// adding +-0 changes nothing.  Runs of the index nmodels (I outside [0, nmodels)): W row 0, K row NaN.
// PAIRS (continuous mode): the rows are (query, model) pairs; row p takes its offset from query row_query[p] and its
// coefficient rows are c_qm = alpha * c_q with alpha = row_scale[p] (one rounded multiply per entry).  A separate
// instantiation, so that the nearest-mode kernels are unchanged.
template <bool UNI, bool PAIRS>
__global__ void __launch_bounds__(OPX_MAX_THREADS, 1) interp_stencil_kernel(InterpStencilParams P) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int nops = P.nops, maxno = P.maxno, opc = P.opc, dim = P.dim;
    double* cs = reinterpret_cast<double*>(smem_raw);                                      // [nops][maxno]
    unsigned long long* nzm = reinterpret_cast<unsigned long long*>(cs + nops * maxno);     // [nops] nonzero slots
    unsigned short* ex = reinterpret_cast<unsigned short*>(nzm + nops);                     // [maxno] slot exponents
    for (int t = threadIdx.x; t < maxno; t += blockDim.x) ex[t] = c_slot_exp.e[dim - 1][t];
    stage_coefficients(P.coef, nops, maxno, cs, nzm);

    // the warp's coefficient rows of one query: cq [opc][maxno], their nonzero slots qnz [opc], Taylor terms tt [3][5]
    double* cq = reinterpret_cast<double*>(smem_raw) + P.cq_off + (size_t)warp * P.cq_doubles;
    unsigned long long* qnz = reinterpret_cast<unsigned long long*>(cq + opc * maxno);
    double* tt = reinterpret_cast<double*>(qnz + opc);

    // units: the runs, whose number the sort left on the device
    const double* ring = reinterpret_cast<double*>(smem_raw) + P.ring_off + (size_t)warp * P.stages * P.stage_doubles;
    WarpRing R(smem_u32(ring), smem_u32(smem_raw + P.bar_off_bytes) + (uint32_t)(warp * P.stages) * 8u, P.stages,
               (uint32_t)P.stage_doubles * 8u, 0, *P.nruns);
    auto issue = [&](uint32_t st, uint32_t bar, long long r) {   // lane 0 only
        const long long c = P.run_case[r];
        uint32_t b = 0;
        CaseMeta m{};
        if (c < P.nmodels) {
            m = case_meta<UNI>(P.meta, P.uni, P.op_stride, c);
            b = op_block_bytes(m);
        }
        mbar_expect_tx_u32(bar, b);
        if (b) tma_load_1d_u32(st, P.op + m.op_off, b, bar);
    };
    R.start(lane, issue);

    long long r = R.first;
    for (long long i = 0; i < R.n_my; ++i, r += R.stride) {
        R.refill(lane, i, r, issue);
        const long long c = P.run_case[r];
        const int q0 = P.run_off[r], nq = P.run_len[r];
        const double* op = ring + (size_t)R.stage * P.stage_doubles;
        R.wait();
        if (c >= P.nmodels) {
            // no model: W row 0, K row NaN (interpolate's NaN for such a query), nothing folded
            for (int t = 0; t < nq; ++t) {
                const long long q = P.perm[q0 + t];
                for (int o = 0; o < nops; ++o) {
                    for (int k = lane; k < P.maxnk; k += 32) P.W[((long long)o * P.nx + q) * P.maxnk + k] = 0.0;
                    if (P.K)
                        for (int s = lane; s < maxno; s += 32)
                            P.K[((long long)o * P.nx + q) * maxno + s] = __longlong_as_double(0x7ff8000000000000LL);
                    if (P.kf && lane == 0) P.kf[(long long)o * P.nx + q] = 0.0;
                }
            }
        } else {
            const CaseMeta m = case_meta<UNI>(P.meta, P.uni, P.op_stride, c);
            for (int t = 0; t < nq; ++t) {
                const long long q = P.perm[q0 + t];
                const long long xq = PAIRS ? (long long)P.row_query[q] : q;
                if (lane < 3) {     // Taylor terms of axis `lane` (h = 0 beyond the dimension: 1, 0, 0, 0, 0)
                    const double h = lane < dim ? P.x[xq * P.x_s0 + lane] - P.xi[c * dim + lane] : 0.0;
                    const Steps st = steps_of(h);
                    double tv = 1.0;
                    tt[lane * 5] = tv;
#pragma unroll
                    for (int n = 1; n < 5; ++n) {
                        tv = __dmul_rn(tv, st.s[n - 1]);
                        tt[lane * 5 + n] = tv;
                    }
                }
                __syncwarp();
                for (int o0 = 0; o0 < nops; o0 += opc) {
                    const int oc = min(opc, nops - o0);
                    for (int idx = lane; idx < oc * maxno; idx += 32) {
                        const int o = idx / maxno, s = idx - o * maxno;
                        const int es = ex[s], a = es & 15, b = (es >> 4) & 15, cz = es >> 8;
                        const double* co = cs + (o0 + o) * maxno;
                        double acc = 0.0;
                        for (unsigned long long bits = nzm[o0 + o]; bits; bits &= bits - 1) {
                            const int D = __ffsll((long long)bits) - 1;
                            const int ed = ex[D], p = ed & 15, pr = (ed >> 4) & 15, pu = ed >> 8;
                            if (a >= p && b >= pr && cz >= pu) {
                                const double T = __dmul_rn(__dmul_rn(tt[a - p], tt[5 + b - pr]), tt[10 + cz - pu]);
                                acc = __dadd_rn(acc, __dmul_rn(co[D], T));
                            }
                        }
                        cq[idx] = PAIRS ? __dmul_rn(P.row_scale[q], acc) : acc;
                    }
                    __syncwarp();
                    for (int o = 0; o < oc; ++o) {
                        const unsigned long long nz = nonzero_slots(cq + o * maxno, maxno, lane);
                        if (lane == 0) qnz[o] = nz;
                    }
                    __syncwarp();
                    contract_case(op, m, cq, qnz, oc, maxno, P.maxnk, P.nx, q, P.W + (long long)o0 * P.nx * P.maxnk,
                                  P.K ? P.K + (long long)o0 * P.nx * maxno : nullptr, P.kf ? P.kf + (long long)o0 * P.nx : nullptr,
                                  lane);
                    __syncwarp();   // cq / qnz / tt are rewritten for the next pass or query
                }
            }
        }
        R.release();
    }
}

template <bool UNI, bool PAIRS>
static cudaError_t launch_interp_stencils_t(const InterpStencilParams& P, int blocks, int threads, size_t smem, cudaStream_t st) {
    const cudaError_t e = cudaFuncSetAttribute(interp_stencil_kernel<UNI, PAIRS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    interp_stencil_kernel<UNI, PAIRS><<<blocks, threads, smem, st>>>(P);
    return cudaGetLastError();
}

cudaError_t launch_interp_stencils(const InterpStencilParams& P, int blocks, int threads, size_t smem, cudaStream_t st) {
    const bool uni = P.meta == nullptr || P.geom_uniform;
    if (P.row_query)
        return uni ? launch_interp_stencils_t<true, true>(P, blocks, threads, smem, st)
                   : launch_interp_stencils_t<false, true>(P, blocks, threads, smem, st);
    return uni ? launch_interp_stencils_t<true, false>(P, blocks, threads, smem, st)
               : launch_interp_stencils_t<false, false>(P, blocks, threads, smem, st);
}

// ---- continuous-mode interpolation operators --------------------------------------------------------------------
// Per query q (one thread): its pairs p in [pair_ptr[q], pair_ptr[q+1]) (models J32[p], ascending), d2 recomputed by the
// ball rule of wlsqm_grid_ball_* (xi - x per axis, square, sum in axis order, each rounded on its own), the weight
// w = (1 - sqrt(d2 / r2))^2 with every operation rounded on its own, S = the sum of w in pair order from +0, and
// alpha[p] = w / S (NaN when S = 0: every member at exactly r).  Also widens J and records each pair's query.
template <int DIM>
__global__ void cont_weights_kernel(const double* __restrict__ x, long long x_s0, const double* __restrict__ xi,
                                    long long nx, double r, const long long* __restrict__ pair_ptr,
                                    const int32_t* __restrict__ J32, long long* __restrict__ J, int* __restrict__ pair_query,
                                    double* __restrict__ alpha) {
    const double r2 = __dmul_rn(r, r);
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < nx; q += (long long)gridDim.x * blockDim.x) {
        const long long p0 = pair_ptr[q], p1 = pair_ptr[q + 1];
        double xq[DIM];
#pragma unroll
        for (int d = 0; d < DIM; ++d) xq[d] = x[q * x_s0 + d];
        double S = 0.0;
        for (long long p = p0; p < p1; ++p) {
            const long long m = J32[p];
            double d2 = 0.0;
#pragma unroll
            for (int d = 0; d < DIM; ++d) {
                const double dd = __dsub_rn(xi[m * DIM + d], xq[d]);
                d2 = __dadd_rn(d2, __dmul_rn(dd, dd));
            }
            const double tmp = __dsub_rn(1.0, __dsqrt_rn(__ddiv_rn(d2, r2)));
            const double w = __dmul_rn(tmp, tmp);
            S = __dadd_rn(S, w);
            alpha[p] = w;
            J[p] = m;
            pair_query[p] = (int)q;
        }
        for (long long p = p0; p < p1; ++p) alpha[p] = __ddiv_rn(alpha[p], S);
    }
}

static unsigned grid_for(long long n, int threads) {
    return (unsigned)std::max<long long>(1, std::min<long long>((n + threads - 1) / threads, 148LL * 32));
}

cudaError_t launch_cont_weights(const double* x, long long x_s0, int dim, const double* xi, long long nx, double r,
                                const long long* pair_ptr, const int32_t* J32, long long* J, int* pair_query, double* alpha,
                                cudaStream_t st) {
    const unsigned b = grid_for(nx, 128);
    if (dim == 1) cont_weights_kernel<1><<<b, 128, 0, st>>>(x, x_s0, xi, nx, r, pair_ptr, J32, J, pair_query, alpha);
    else if (dim == 2) cont_weights_kernel<2><<<b, 128, 0, st>>>(x, x_s0, xi, nx, r, pair_ptr, J32, J, pair_query, alpha);
    else cont_weights_kernel<3><<<b, 128, 0, st>>>(x, x_s0, xi, nx, r, pair_ptr, J32, J, pair_query, alpha);
    return cudaGetLastError();
}

// *flag := 1 where a[i] != b[i], i < n
__global__ void ptr_mismatch_kernel(const long long* __restrict__ a, const long long* __restrict__ b, long long n, int* flag) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        if (a[i] != b[i]) *flag = 1;
}

cudaError_t launch_ptr_mismatch(const long long* a, const long long* b, long long n, int* flag, cudaStream_t st) {
    ptr_mismatch_kernel<<<grid_for(n, 256), 256, 0, st>>>(a, b, n, flag);
    return cudaGetLastError();
}

// Candidate slot (p, k) of pair p (model m = J[p]), k < L = max nk + 1: k < nk_m the neighbour hoods[m][k], k = L - 1
// the folded known F (column center + m) when centre folding applies to m, else no column.
__device__ __forceinline__ unsigned cont_slot_column(const ContCsrParams& P, long long p, int k) {
    const long long m = P.J[p];
    const CaseMeta cm = P.meta ? P.meta[m] : P.uni;
    if (k < cm.nk) return (unsigned)P.hoods[m * P.hoods_s0 + k];
    if (k == P.L - 1 && P.center >= 0 && (cm.knowns & 1LL)) return (unsigned)(P.center + m);
    return CONT_NO_COLUMN;
}
__device__ __forceinline__ double cont_slot_value(const ContCsrParams& P, int o, long long p, int k) {
    return k < P.maxnk ? P.W[((long long)o * P.npairs + p) * P.maxnk + k] : P.kf[(long long)o * P.npairs + p];
}
__device__ __forceinline__ long long cont_row_slots(const ContCsrParams& P, long long q) {
    return (P.pair_ptr[q + 1] - P.pair_ptr[q]) * P.L;
}

// Short rows (at most row_cap candidate slots): one warp per query stages the keys (column << 32 | slot) of its slots in
// shared memory and sorts them (bitonic, padded to a power of two with ~0).  Keys are unique, so equal columns end up
// adjacent in slot order -- the candidate order.  FILL = false: the number of distinct columns -> cnt[q]; FILL = true:
// column and per operator the run's values summed from +0 in candidate order at rp[q] + (the run's rank).  Longer rows
// are left to the sort route below.
template <bool FILL, typename IDX>
__global__ void __launch_bounds__(CONT_ROW_WARPS * 32) cont_row_kernel(ContCsrParams P) {
    extern __shared__ unsigned long long cont_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    unsigned long long* buf = cont_smem + (size_t)warp * P.row_cap;
    const long long GW = (long long)gridDim.x * nwarps;
    for (long long q = (long long)blockIdx.x * nwarps + warp; q < P.nx; q += GW) {
        const long long nl = cont_row_slots(P, q);
        if (nl > P.row_cap) continue;
        const long long p0 = P.pair_ptr[q];
        const int n = (int)nl;
        int N = 32;
        while (N < n) N <<= 1;
        for (int i = lane; i < N; i += 32) {
            unsigned long long key = ~0ull;
            if (i < n) {
                const int pp = i / P.L;
                const unsigned c = cont_slot_column(P, p0 + pp, i - pp * P.L);
                if (c != CONT_NO_COLUMN) key = ((unsigned long long)c << 32) | (unsigned)i;
            }
            buf[i] = key;
        }
        __syncwarp();
        for (int size = 2; size <= N; size <<= 1)
            for (int stride = size >> 1; stride > 0; stride >>= 1) {
                for (int t = lane; t < (N >> 1); t += 32) {
                    const int a = ((t & ~(stride - 1)) << 1) | (t & (stride - 1)), b = a + stride;
                    const unsigned long long ka = buf[a], kb = buf[b];
                    if ((ka > kb) == ((a & size) == 0)) { buf[a] = kb; buf[b] = ka; }
                }
                __syncwarp();
            }
        long long cnt = 0;
        const long long base = FILL ? P.rp[q] : 0;
        for (int i0 = 0; i0 < n; i0 += 32) {
            const int i = i0 + lane;
            unsigned long long key = ~0ull;
            bool head = false;
            if (i < n) {
                key = buf[i];
                head = key != ~0ull && (i == 0 || (key >> 32) != (buf[i - 1] >> 32));
            }
            const unsigned bal = __ballot_sync(0xffffffffu, head);
            if (FILL && head) {
                const long long pos = base + cnt + __popc(bal & ((1u << lane) - 1u));
                const unsigned c = (unsigned)(key >> 32);
                static_cast<IDX*>(P.col)[pos] = (IDX)c;
                for (int o = 0; o < P.nops; ++o) {
                    double v = 0.0;
                    for (int j = i; j < n && (unsigned)(buf[j] >> 32) == c; ++j) {
                        const int sl = (int)(unsigned)buf[j], pp = sl / P.L;
                        v = __dadd_rn(v, cont_slot_value(P, o, p0 + pp, sl - pp * P.L));
                    }
                    P.values[(long long)o * P.nnz + pos] = v;
                }
            }
            cnt += __popc(bal);
        }
        if (!FILL && lane == 0) P.cnt[q] = cnt;
        __syncwarp();   // buf is rewritten for the next row
    }
}

// ---- sort route for rows longer than row_cap: chunk [q0, q1) of the queries, slots [slot0, slot0 + nslots) -------
// chunk slot i (global slot g = slot0 + i, pair g / L): its column when its row is long, else none (sorted last)
__global__ void cont_keys_kernel(ContCsrParams P) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < P.nslots; i += (long long)gridDim.x * blockDim.x) {
        const long long g = P.slot0 + i, p = g / P.L;
        const bool lng = cont_row_slots(P, P.pair_query[p]) > P.row_cap;
        P.keys[i] = lng ? cont_slot_column(P, p, (int)(g - p * P.L)) : CONT_NO_COLUMN;
        P.cand[i] = (int)i;
    }
}

// seg[j] = the first chunk slot of query q0 + j, j <= q1 - q0
__global__ void cont_seg_kernel(ContCsrParams P) {
    for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j <= P.q1 - P.q0; j += (long long)gridDim.x * blockDim.x)
        P.seg[j] = (int)(P.pair_ptr[P.q0 + j] * P.L - P.slot0);
}

// head[i] = 1 where sorted chunk slot i starts a (query, column) run; head[nslots] = 0 (the scan's total)
__global__ void cont_heads_kernel(ContCsrParams P) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i <= P.nslots; i += (long long)gridDim.x * blockDim.x) {
        int h = 0;
        if (i < P.nslots) {
            const unsigned key = P.keys_sorted[i];
            const bool first = i == 0 || P.pair_query[(P.slot0 + i) / P.L] != P.pair_query[(P.slot0 + i - 1) / P.L];
            h = key != CONT_NO_COLUMN && (first || key != P.keys_sorted[i - 1]);
        }
        P.head[i] = h;
    }
}

// count: cnt[q] of the chunk's long rows
__global__ void cont_long_count_kernel(ContCsrParams P) {
    for (long long q = P.q0 + (long long)blockIdx.x * blockDim.x + threadIdx.x; q < P.q1; q += (long long)gridDim.x * blockDim.x)
        if (cont_row_slots(P, q) > P.row_cap) P.cnt[q] = P.hpos[P.seg[q - P.q0 + 1]] - P.hpos[P.seg[q - P.q0]];
}

// fill: one thread per run head, the run's values summed in candidate order from +0 (the sort is stable)
template <typename IDX>
__global__ void cont_long_fill_kernel(ContCsrParams P) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < P.nslots; i += (long long)gridDim.x * blockDim.x) {
        if (!P.head[i]) continue;
        const unsigned key = P.keys_sorted[i];
        const long long q = P.pair_query[(P.slot0 + i) / P.L];
        const long long s0 = P.seg[q - P.q0], end = P.seg[q - P.q0 + 1];
        const long long pos = P.rp[q] + P.hpos[i] - P.hpos[s0];
        static_cast<IDX*>(P.col)[pos] = (IDX)key;
        for (int o = 0; o < P.nops; ++o) {
            double v = 0.0;
            for (long long j = i; j < end && P.keys_sorted[j] == key; ++j) {
                const long long g = P.slot0 + P.cand_sorted[j], p = g / P.L;
                v = __dadd_rn(v, cont_slot_value(P, o, p, (int)(g - p * P.L)));
            }
            P.values[(long long)o * P.nnz + pos] = v;
        }
    }
}

// One chunk of the sort route: keys, stable sort per query, heads, scan, then the count or the fill of its long rows.
// tmp == nullptr: *tmp_bytes := the scratch needed for a chunk of P.nslots slots and P.q1 - P.q0 queries.
cudaError_t cont_long_rows(const ContCsrParams& P, bool fill, int index_bits, void* tmp, size_t* tmp_bytes, cudaStream_t st) {
    const int n = (int)P.nslots, nseg = (int)(P.q1 - P.q0);
    if (!tmp) {
        size_t a = 0, b = 0;
        cudaError_t e = cub::DeviceSegmentedSort::StableSortPairs(nullptr, a, P.keys, const_cast<unsigned*>(P.keys_sorted),
                                                                  P.cand, const_cast<int*>(P.cand_sorted), n, nseg, P.seg,
                                                                  P.seg + 1, st);
        if (e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(nullptr, b, P.head, const_cast<int*>(P.hpos), n + 1, st);
        *tmp_bytes = std::max(a, b);
        return e;
    }
    cont_seg_kernel<<<grid_for(nseg + 1, 256), 256, 0, st>>>(P);
    cont_keys_kernel<<<grid_for(n, 256), 256, 0, st>>>(P);
    cudaError_t e = cudaGetLastError();
    size_t tb = *tmp_bytes;
    if (e == cudaSuccess)
        e = cub::DeviceSegmentedSort::StableSortPairs(tmp, tb, P.keys, const_cast<unsigned*>(P.keys_sorted), P.cand,
                                                      const_cast<int*>(P.cand_sorted), n, nseg, P.seg, P.seg + 1, st);
    if (e == cudaSuccess) {
        cont_heads_kernel<<<grid_for(n + 1, 256), 256, 0, st>>>(P);
        e = cudaGetLastError();
    }
    tb = *tmp_bytes;
    if (e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(tmp, tb, P.head, const_cast<int*>(P.hpos), n + 1, st);
    if (e != cudaSuccess) return e;
    if (!fill) cont_long_count_kernel<<<grid_for(nseg, 256), 256, 0, st>>>(P);
    else if (index_bits == 32) cont_long_fill_kernel<int32_t><<<grid_for(n, 256), 256, 0, st>>>(P);
    else cont_long_fill_kernel<long long><<<grid_for(n, 256), 256, 0, st>>>(P);
    return cudaGetLastError();
}

template <bool FILL, typename IDX>
static cudaError_t launch_cont_row_t(const ContCsrParams& P, cudaStream_t st) {
    const size_t smem = (size_t)CONT_ROW_WARPS * P.row_cap * 8;
    const cudaError_t e = cudaFuncSetAttribute(cont_row_kernel<FILL, IDX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const unsigned blocks = (unsigned)std::max<long long>(1, std::min<long long>((P.nx + CONT_ROW_WARPS - 1) / CONT_ROW_WARPS, 148LL * 64));
    cont_row_kernel<FILL, IDX><<<blocks, CONT_ROW_WARPS * 32, smem, st>>>(P);
    return cudaGetLastError();
}

// rowptr[q] = rp[q], q <= nx
template <typename IDX>
__global__ void cont_rowptr_kernel(ContCsrParams P) {
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q <= P.nx; q += (long long)gridDim.x * blockDim.x)
        static_cast<IDX*>(P.rowptr)[q] = (IDX)P.rp[q];
}

// the short rows: count (fill = false) or rowptr and fill
cudaError_t launch_cont_rows(const ContCsrParams& P, bool fill, int index_bits, cudaStream_t st) {
    if (fill) {
        if (index_bits == 32) cont_rowptr_kernel<int32_t><<<grid_for(P.nx + 1, 256), 256, 0, st>>>(P);
        else cont_rowptr_kernel<long long><<<grid_for(P.nx + 1, 256), 256, 0, st>>>(P);
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    if (P.row_cap == 0) return cudaSuccess;
    if (!fill) return launch_cont_row_t<false, int32_t>(P, st);
    return index_bits == 32 ? launch_cont_row_t<true, int32_t>(P, st) : launch_cont_row_t<true, long long>(P, st);
}

// keys[q] = I[q] when it is a case index, else nmodels; qidx[q] = q
__global__ void interp_keys_kernel(const long long* __restrict__ I, long long nx, long long nmodels, int* __restrict__ keys,
                                   int* __restrict__ qidx) {
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < nx; q += (long long)gridDim.x * blockDim.x) {
        const long long m = I[q];
        keys[q] = (int)(m >= 0 && m < nmodels ? m : nmodels);
        qidx[q] = (int)q;
    }
}

// The runs of equal case index among the queries: a stable radix sort of (key, q) on the bits that keys <= nmodels use,
// then run-length encoding and an exclusive scan of the run lengths.  tmp == nullptr: *tmp_bytes := the scratch needed.
cudaError_t interp_runs(const long long* I, long long nx, long long nmodels, const InterpRuns& R, void* tmp, size_t* tmp_bytes,
                        cudaStream_t st) {
    int end_bit = 1;
    while (end_bit < 32 && (1LL << end_bit) <= nmodels) ++end_bit;
    const int n = (int)nx;
    if (!tmp) {
        size_t a = 0, b = 0, c = 0;
        cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, a, R.keys, R.keys_sorted, R.qidx, R.perm, n, 0, end_bit, st);
        if (e == cudaSuccess) e = cub::DeviceRunLengthEncode::Encode(nullptr, b, R.keys_sorted, R.run_case, R.run_len, R.nruns, n, st);
        if (e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(nullptr, c, R.run_len, R.run_off, n, st);
        *tmp_bytes = std::max(a, std::max(b, c));
        return e;
    }
    const unsigned blocks = (unsigned)std::max<long long>(1, std::min<long long>((nx + 255) / 256, 148LL * 32));
    interp_keys_kernel<<<blocks, 256, 0, st>>>(I, nx, nmodels, R.keys, R.qidx);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemsetAsync(R.run_len, 0, (size_t)nx * sizeof(int), st);
    size_t tb = *tmp_bytes;
    if (e == cudaSuccess) e = cub::DeviceRadixSort::SortPairs(tmp, tb, R.keys, R.keys_sorted, R.qidx, R.perm, n, 0, end_bit, st);
    tb = *tmp_bytes;
    if (e == cudaSuccess) e = cub::DeviceRunLengthEncode::Encode(tmp, tb, R.keys_sorted, R.run_case, R.run_len, R.nruns, n, st);
    tb = *tmp_bytes;
    if (e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(tmp, tb, R.run_len, R.run_off, n, st);
    return e;
}

// One warp per CSR row.  FILL = false: the number of distinct columns of row i -> cnt[i].  FILL = true: columns in
// ascending order at rp[i] ..., each with its W entries summed in ascending k, the folded known-F weight added last.
// A column's rank is the number of distinct columns below it, so no sort is needed: an O(nk^2) comparison per row
// against the indices staged in shared memory (broadcast reads).
// MAP (P.row_case given): row i belongs to case c = row_case[i] -- the neighbour list, record and fold column
// center + c are the case's, W / kf / the output the row's; a case outside [0, nmodels) gives an empty row.
template <bool FILL, typename IDX, bool MAP>
__global__ void __launch_bounds__(CSR_MAX_WARPS * 32) csr_kernel(CsrParams P) {
    extern __shared__ int csr_smem[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int nwarps = blockDim.x >> 5;
    const int mk = max(P.maxnk, 1);
    int* hs = csr_smem + (size_t)warp * mk;                  // the row's used indices
    unsigned char* fl = reinterpret_cast<unsigned char*>(csr_smem + (size_t)nwarps * mk) + (size_t)warp * mk;
                                                              // bit 0: first occurrence, bit 1: occurs again later
    const long long GW = (long long)gridDim.x * nwarps;
    for (long long i = (long long)blockIdx.x * nwarps + warp; i < P.ncases; i += GW) {
        long long c = i;
        bool live = true;
        if (MAP) {
            c = P.row_case[i];
            live = c >= 0 && c < P.nmodels;
            if (!live) c = 0;
        }
        const CaseMeta m = P.meta ? P.meta[c] : P.uni;
        const int nk = live ? m.nk : 0;
        const int32_t* hr = P.hoods + c * P.hoods_s0;
        for (int k = lane; k < nk; k += 32) hs[k] = hr[k];
        __syncwarp();
        const bool fold = live && P.center >= 0 && (m.knowns & 1LL);
        const long long fc = P.center + c;
        int cnt = 0;
        bool fc_in = false;
        for (int k = lane; k - lane < nk; k += 32) {
            int f = 0;
            if (k < nk) {
                const int p = hs[k];
                f = 1;
                for (int t = 0; t < nk; ++t)
                    if (hs[t] == p) {
                        if (t < k) f &= ~1;
                        else if (t > k) f |= 2;
                    }
                if (FILL) fl[k] = (unsigned char)f;
                if (fold && p == fc) fc_in = true;
            }
            cnt += __popc(__ballot_sync(0xffffffffu, f & 1));
        }
        fc_in = __any_sync(0xffffffffu, fc_in);
        const bool extra = fold && !fc_in;
        if (!FILL) {
            if (lane == 0) P.cnt[i] = cnt + (extra ? 1 : 0);
        } else {
            __syncwarp();
            const long long r0 = P.rp[i];
            IDX* col = static_cast<IDX*>(P.col);
            if (lane == 0) {
                static_cast<IDX*>(P.rowptr)[i] = (IDX)r0;
                if (i == P.ncases - 1) static_cast<IDX*>(P.rowptr)[P.ncases] = (IDX)P.rp[P.ncases];
            }
            auto rank_of = [&](long long p) {
                int r = 0;
                for (int t = 0; t < nk; ++t) r += ((fl[t] & 1) && hs[t] < p) ? 1 : 0;
                return r + ((extra && fc < p) ? 1 : 0);
            };
            for (int k = lane; k < nk; k += 32) {
                const int f = fl[k];
                if (!(f & 1)) continue;
                const int p = hs[k];
                const long long pos = r0 + rank_of(p);
                col[pos] = (IDX)p;
                for (int o = 0; o < P.nops; ++o) {
                    const double* w = P.W + ((long long)o * P.ncases + i) * P.maxnk;
                    double v = w[k];
                    if (f & 2)
                        for (int t = k + 1; t < nk; ++t)
                            if (hs[t] == p) v += w[t];
                    if (fold && p == fc) v += P.kf[(long long)o * P.ncases + i];
                    P.values[(long long)o * P.nnz + pos] = v;
                }
            }
            if (extra && lane == 0) {
                const long long pos = r0 + rank_of(fc);
                col[pos] = (IDX)fc;
                for (int o = 0; o < P.nops; ++o) P.values[(long long)o * P.nnz + pos] = P.kf[(long long)o * P.ncases + i];
            }
        }
        __syncwarp();   // the row's staged indices are read until here
    }
}

// As many warps per CTA (up to 8) as shared memory holds rows of max nk: CSR_BYTES_PER_NK bytes per neighbour and warp
template <typename Kernel>
static cudaError_t launch_csr(Kernel kernel, const CsrParams& P, cudaStream_t st) {
    const size_t per_warp = (size_t)CSR_BYTES_PER_NK * std::max(P.maxnk, 1);
    const int warps = (int)std::min<size_t>(CSR_MAX_WARPS, CSR_SMEM_MAX / per_warp);
    if (warps < 1) return cudaErrorInvalidValue;     // (the caller refuses such batches first)
    const size_t smem = (size_t)warps * per_warp;
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const unsigned blocks = (unsigned)std::max<long long>(1, std::min<long long>((P.ncases + warps - 1) / warps, 148LL * 64));
    kernel<<<blocks, warps * 32, smem, st>>>(P);
    return cudaGetLastError();
}

cudaError_t launch_csr_count(const CsrParams& P, cudaStream_t st) {
    return P.row_case ? launch_csr(csr_kernel<false, int, true>, P, st) : launch_csr(csr_kernel<false, int, false>, P, st);
}

cudaError_t csr_scan(long long* cnt, long long* rp, long long n1, void* tmp, size_t* tmp_bytes, cudaStream_t st) {
    return cub::DeviceScan::ExclusiveSum(tmp, *tmp_bytes, cnt, rp, (int)n1, st);
}

cudaError_t launch_csr_fill(const CsrParams& P, int index_bits, cudaStream_t st) {
    if (P.row_case)
        return index_bits == 32 ? launch_csr(csr_kernel<true, int32_t, true>, P, st) : launch_csr(csr_kernel<true, long long, true>, P, st);
    return index_bits == 32 ? launch_csr(csr_kernel<true, int32_t, false>, P, st) : launch_csr(csr_kernel<true, long long, false>, P, st);
}

}  // namespace wlsqm
