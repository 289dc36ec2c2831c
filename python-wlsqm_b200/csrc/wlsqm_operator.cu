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
template <bool UNI>
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
                if (lane < 3) {     // Taylor terms of axis `lane` (h = 0 beyond the dimension: 1, 0, 0, 0, 0)
                    const double h = lane < dim ? P.x[q * P.x_s0 + lane] - P.xi[c * dim + lane] : 0.0;
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
                        cq[idx] = acc;
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

cudaError_t launch_interp_stencils(const InterpStencilParams& P, int blocks, int threads, size_t smem, cudaStream_t st) {
    const bool uni = P.meta == nullptr || P.geom_uniform;
    cudaError_t e;
    if (uni) {
        e = cudaFuncSetAttribute(interp_stencil_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        interp_stencil_kernel<true><<<blocks, threads, smem, st>>>(P);
    } else {
        e = cudaFuncSetAttribute(interp_stencil_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        interp_stencil_kernel<false><<<blocks, threads, smem, st>>>(P);
    }
    return cudaGetLastError();
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
