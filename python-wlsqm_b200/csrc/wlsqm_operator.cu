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
// stencil_kernel: one warp per case streams its block into a shared-memory ring with the bulk copies of
// solve_kernel (same CaseMeta addressing, case_meta / op_block_bytes in wlsqm_kernels.h) and produces all nops
// operators from that one read; the coefficients live in shared memory.  Bound by the HBM read of the blocks.
// csr_kernel<false>: distinct columns per row (count); cub exclusive scan; csr_kernel<true>: columns in ascending
// order, merged values (fill).  A warp per row; the row's used hood indices are staged in shared memory.
#include <cub/cub.cuh>
#include "wlsqm_common.cuh"
#include "wlsqm_kernels.h"

namespace wlsqm {

constexpr int OPX_MAX_THREADS = 1024;
constexpr int CSR_MAX_WARPS = 8;

template <bool UNI>
__global__ void __launch_bounds__(OPX_MAX_THREADS, 1) stencil_kernel(StencilParams P) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int nwarps = blockDim.x >> 5;
    const int nops = P.nops, maxno = P.maxno;
    double* cs = reinterpret_cast<double*>(smem_raw);                                      // [nops][maxno]
    unsigned long long* nzm = reinterpret_cast<unsigned long long*>(cs + nops * maxno);     // [nops] nonzero slots
    for (int t = threadIdx.x; t < nops * maxno; t += blockDim.x) cs[t] = P.coef[t];
    __syncthreads();
    for (int o = warp; o < nops; o += nwarps) {
        const double* co = cs + o * maxno;
        const unsigned lo = __ballot_sync(0xffffffffu, lane < maxno && co[lane] != 0.0);
        const unsigned hi = __ballot_sync(0xffffffffu, lane + 32 < maxno && co[lane + 32] != 0.0);
        if (lane == 0) nzm[o] = ((unsigned long long)hi << 32) | lo;
    }
    __syncthreads();

    const int S = P.stages;
    double* ring = reinterpret_cast<double*>(smem_raw) + P.ring_off + (size_t)warp * S * P.stage_doubles;
    const uint32_t ring_u32 = smem_u32(ring);
    const uint32_t bars_u32 = smem_u32(smem_raw + P.bar_off_bytes) + (uint32_t)(warp * S) * 8u;
    const uint32_t stage_bytes = (uint32_t)P.stage_doubles * 8u;
    const long long gw = (long long)blockIdx.x * nwarps + warp;
    const long long GW = (long long)gridDim.x * nwarps;
    const long long n_my = gw < P.ncases ? (P.ncases - gw + GW - 1) / GW : 0;

    auto issue = [&](int s, long long c) {   // lane 0 only
        const CaseMeta m = case_meta<UNI>(P.meta, P.uni, P.op_stride, c);
        const uint32_t st = ring_u32 + (uint32_t)s * stage_bytes, bar = bars_u32 + (uint32_t)s * 8u;
        const uint32_t b = op_block_bytes(m);
        mbar_expect_tx_u32(bar, b);
        if (b) tma_load_1d_u32(st, P.op + m.op_off, b, bar);
    };
    if (lane == 0) {
        for (int s = 0; s < S; ++s) mbar_init_u32(bars_u32 + (uint32_t)s * 8u, 1);
        fence_mbar_init();
        for (int s = 0; s < S - 1 && s < n_my; ++s) issue(s, gw + (long long)s * GW);
    }
    __syncwarp();

    int stage = 0;
    uint32_t phase = 0;
    long long c = gw;
    for (long long i = 0; i < n_my; ++i, c += GW) {
        if (lane == 0 && i + S - 1 < n_my) {
            int sn = stage + S - 1;
            if (sn >= S) sn -= S;
            issue(sn, c + (long long)(S - 1) * GW);
        }
        const CaseMeta m = case_meta<UNI>(P.meta, P.uni, P.op_stride, c);
        const int nk = m.nk, no = m.no, nr = m.nr;
        const unsigned long long knowns = (unsigned long long)m.knowns;
        const unsigned long long unk = ~knowns & ((1ull << no) - 1);     // no <= 35
        const double* op = ring + (size_t)stage * P.stage_doubles;
        mbar_wait_u32(bars_u32 + (uint32_t)stage * 8u, phase);

        // sum over the unknown slots with a nonzero coefficient, ascending, of c[s] * row[j(s)]
        auto contract = [&](const double* co, unsigned long long bits, const double* row) {
            double acc = 0.0;
            for (; bits; bits &= bits - 1) {
                const int s = __ffsll((long long)bits) - 1;
                const int j = s - __popcll(knowns & ((1ull << s) - 1));
                acc = fma(co[s], row[j], acc);
            }
            return acc;
        };
        // neighbour rows: lane = k
        for (int k = lane; k < P.maxnk; k += 32) {
            const double* row = op + k * nr;
            double* w = P.W + c * P.maxnk + k;
            for (int o = 0; o < nops; ++o) {
                const double v = k < nk ? contract(cs + o * maxno, nzm[o] & unk, row) : 0.0;
                w[(long long)o * P.ncases * P.maxnk] = v;
            }
        }
        // known slots: lane = slot m, its row is nk + (its position among the knowns)
        if (P.K || P.kf) {
            for (int s = lane; s < maxno; s += 32) {
                const bool kn = s < no && ((knowns >> s) & 1ull);
                const double* row = op + (nk + __popcll(knowns & ((1ull << s) - 1))) * nr;
                for (int o = 0; o < nops; ++o) {
                    double v = 0.0;
                    if (kn) v = contract(cs + o * maxno, nzm[o] & unk, row) + cs[o * maxno + s];
                    if (P.kf && s == 0) {
                        P.kf[(long long)o * P.ncases + c] = v;   // folded into column center + c of the CSR row
                        v = 0.0;
                    }
                    if (P.K) P.K[((long long)o * P.ncases + c) * maxno + s] = v;
                }
            }
        }
        __syncwarp();   // every lane is done with this stage before lane 0 re-arms it
        if (++stage == S) { stage = 0; phase ^= 1u; }
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

// One warp per CSR row.  FILL = false: the number of distinct columns of row i -> cnt[i].  FILL = true: columns in
// ascending order at rp[i] ..., each with its W entries summed in ascending k, the folded known-F weight added last.
// A column's rank is the number of distinct columns below it, so no sort is needed: an O(nk^2) comparison per row
// against the indices staged in shared memory (broadcast reads).
template <bool FILL, typename IDX>
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
        const CaseMeta m = P.meta ? P.meta[i] : P.uni;
        const int nk = m.nk;
        const int32_t* hr = P.hoods + i * P.hoods_s0;
        for (int k = lane; k < nk; k += 32) hs[k] = hr[k];
        __syncwarp();
        const bool fold = P.center >= 0 && (m.knowns & 1LL);
        const long long fc = P.center + i;
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

cudaError_t launch_csr_count(const CsrParams& P, cudaStream_t st) { return launch_csr(csr_kernel<false, int>, P, st); }

cudaError_t csr_scan(long long* cnt, long long* rp, long long n1, void* tmp, size_t* tmp_bytes, cudaStream_t st) {
    return cub::DeviceScan::ExclusiveSum(tmp, *tmp_bytes, cnt, rp, (int)n1, st);
}

cudaError_t launch_csr_fill(const CsrParams& P, int index_bits, cudaStream_t st) {
    return index_bits == 32 ? launch_csr(csr_kernel<true, int32_t>, P, st) : launch_csr(csr_kernel<true, long long>, P, st);
}

}  // namespace wlsqm
