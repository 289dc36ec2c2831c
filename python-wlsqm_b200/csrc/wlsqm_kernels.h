// wlsqm_kernels.h -- parameter blocks and launchers shared by the kernels and the C-ABI layer.
#pragma once
#include <cuda_runtime.h>
#include "wlsqm_common.cuh"

namespace wlsqm {

constexpr int PREP_MAX_THREADS = 512;        // shared-memory variant (wlsqm_prepare_smem.cu)
constexpr int PREP_REG_SMALL_THREADS = 1024; // ... models of at most 8 DOFs: 64 registers, as many warps as shared memory holds
constexpr int PREP_REG_MAX_THREADS = 640;    // largest launch bound among the instantiations (2D order 4: 20 warps at 96 registers)
constexpr int PREP_REG_THREADS = 512;        // register/DMMA variant (wlsqm_prepare.cu): launch bound; the host picks the CTA size
constexpr int WLSQM_MAX_PEERS = 8;           // GPUs of one NVSwitch domain that can receive the fused gather
constexpr int PREP_CB = 36;                  // row stride (doubles) inside a 32-column block of the monomial table
constexpr int SOLVE_MAX_THREADS = 1024;       // ALGO_BASIC variants (<= 64 registers per thread)
constexpr int SOLVE_MAX_THREADS_ITER = 512;   // ALGO_ITERATIVE variants carry the Taylor evaluator
constexpr int SOLVE_ITER12_THREADS = 768;     // ... in 1D / 2D: one 24-warp CTA per SM (80 registers)

// All strides are in elements (doubles), all offsets into per-warp shared memory in doubles.
struct PrepareParams {
    const CaseMeta* meta;   // per-case records, or nullptr when the batch is uniform
    CaseMeta uni;           // the uniform record (op_off ignored)
    long long op_stride;    // uniform batches: doubles per operator block
    long long ncases;
    const double* xi; long long xi_s0;               // [ncases][dim]
    const double* xk; long long xk_s0, xk_s1;        // [ncases][nk][dim], last axis contiguous
    double* op;                                      // operator blocks (output)
    double* As; int as_stride;                       // debug: scaled matrices [ncases][as_stride] or nullptr
    int warp_doubles, off_w, off_a, off_rs, off_s, off_i;
};

// register/DMMA prepare kernel (wlsqm_prepare.cu)
struct PrepRegParams {
    const CaseMeta* meta;   // per-case records, or nullptr when the batch is uniform
    CaseMeta uni;
    long long op_stride;
    long long ncases;
    const double* xi; long long xi_s0;               // [ncases][dim]
    const double* xk; long long xk_s0, xk_s1;        // [ncases][nk][dim], last axis contiguous
    double* op;                                      // operator blocks (output)
    double* As; int as_stride;                       // debug: scaled matrices [ncases][as_stride] or nullptr
    int geom_uniform;                                // every case has the sizes of `uni`; only meta[c].knowns is read
    int nb;                                          // 32-column blocks of the monomial table
    int fit_doubles;                                 // shared-memory doubles per fit region (prep_reg_fit_doubles)
    int warp_doubles;                                // per warp: monomial table + prep_reg_fits_per_warp() fit regions
    // one-shot fit (no operator): data and in/out solution; fk == nullptr selects the operator-building kernel
    const double* fk; long long fk_s0, fk_s1;        // [ncases][nk]
    double* fi; long long fi_s0;                     // [ncases][>= no]: knowns read, unknowns written
    int phase_sync;                                  // CTA barrier at every phase boundary (instruction-cache sharing)
    const int* perm;                                 // launch over a case list: entry v of [0, ncases) is case perm[v] (nullptr: v)
};

struct SolveParams {
    const CaseMeta* meta;
    CaseMeta uni;
    int geom_uniform;                                // every case has the sizes of `uni`; only meta[c].knowns is read
    long long op_stride;
    long long ncases;                                // cases [case_lo, ncases) are processed by this launch
    long long case_lo;
    const double* op;
    const double* fk; long long fk_s0, fk_s1;        // [ncases][nk] fully strided (simple.pyx:149-159)
    const double* fi_in; long long fi_in_s0;         // caller's fi (known values are read from it)
    double* fi_case; int fi_case_ld;                 // solver-owned copy of the solution (Case.fi)
    double* fi_out; long long fi_out_s0;             // caller's fi on the device, or nullptr (deferred write-back)
    double* sens; long long sens_s0, sens_s1;        // [ncases][nk][no], last axis contiguous, or nullptr
    int algorithm, max_iter;
    const double* xi; long long xi_s0;               // ALGO_ITERATIVE: geometry kept at prepare()
    const double* xk; long long xk_s0, xk_s1;
    int* iters_max;                                  // max refinement iterations over all cases
    int* iters_case;                                 // optional per-case iteration counts
    int stages, stage_doubles;                       // TMA ring per warp; a stage is [operator | fext | xk]
    int off_f, off_xk;                               // offsets of fext / xk inside a stage (doubles)
    int warp_doubles, off_fi, off_r;                 // per-warp smem carve-up (doubles)
    int bar_off_bytes;                               // start of the mbarrier array
    int f_tma, xk_tma;                               // fk / xk rows qualify for bulk copies (alignment, unit stride)
    int pack_lw;                                     // packed variant: log2 of the lanes per case
    // fused result gather (multi-GPU, SURVEY.md 8e): every solved row is also stored into the global solution array of
    // each of `ngather` GPUs (this one included) through peer memory over NVLink -- the all-gather of fi without a
    // collective: row c of this solver is row gather_row0 + c there
    int ngather;
    double* gather[WLSQM_MAX_PEERS];
    long long gather_row0, gather_s0;
    int gather_full;                                 // rows are whole 128 B lines (gather_s0 a multiple of 16, <= 32): the padding is stored too
};

// Field-batched solve (wlsqm_solve.cu): the nf fields of a pass share each streamed operator block.  Field f reads its
// data at P.fk + f * fk_sf (strides P.fk_s0 / P.fk_s1) and its known values from fi + f * fi_sf (row stride fi_s0), and
// writes its unknown slots there.  A stage of P's ring is [operator | fext of field 0 | ... | fext of field nf-1 | xk]:
// the fext slots are f_doubles apart from P.off_f on, xk is at P.off_xk (packed variant: [CPW operator blocks | CPW fk
// rows of each field, f_doubles apart | CPW x nkn known values of each field, k_doubles apart from P.off_xk]).
// P.fi_in / fi_out / fi_case / sens / gather are not used; P.iters_case[c] is raised to the maximum over the fields.
constexpr int SOLVE_FIELDS_THREADS = 512;     // field kernels: 128 registers hold the accumulators of 8 fields
constexpr int SOLVE_FIELDS_BLOCK = 8;         // fields fed by one shared-memory read of an operator element
struct FieldsParams {
    SolveParams P;
    int nf, f_doubles, k_doubles;
    long long fk_sf;
    double* fi; long long fi_s0, fi_sf;
};

// operator export (wlsqm_operator.cu): contraction of the operator blocks with coefficient rows, CSR assembly
struct StencilParams {
    const CaseMeta* meta;
    CaseMeta uni;
    int geom_uniform;                                // every case has the sizes of `uni`; only meta[c].knowns is read
    long long op_stride;
    long long ncases;
    const double* op;
    const double* coef;                              // [nops][maxno] (device copy of the caller's coefficients)
    int nops, maxnk, maxno;
    double* W;                                       // [nops][ncases][maxnk]
    double* K;                                       // [nops][ncases][maxno] or nullptr
    double* kf;                                      // centre folding: [nops][ncases] known-F weight (K[.][.][0] := 0), or nullptr
    int stages, stage_doubles, ring_off, bar_off_bytes;   // per-warp ring of operator blocks (doubles / bytes)
};

// CSR assembly stages a row's used hood indices (int) and a flag byte per index in shared memory: max nk is bounded by
// CSR_SMEM_MAX / CSR_BYTES_PER_NK (46 489), above what prepare accepts (both prepare kernels stage >= 8 bytes per neighbour)
constexpr int CSR_BYTES_PER_NK = 5;
constexpr size_t CSR_SMEM_MAX = 227 * 1024;
struct CsrParams {
    const CaseMeta* meta;
    CaseMeta uni;
    long long ncases;                                // rows: the cases, or the queries when row_case is given
    const long long* row_case;                       // case of each row (interpolation operators), or nullptr: row i is case i;
    long long nmodels;                               //   a case outside [0, nmodels) gives an empty row
    const int32_t* hoods; int hoods_s0;              // [cases][hoods_s0], only the first nk_c of case c are read
    long long center;                                // column of case 0's own point, or -1 (no folding)
    int maxnk;
    long long* cnt;                                  // count pass: distinct columns of row i
    const long long* rp;                             // fill pass: exclusive scan of cnt, [ncases + 1]
    const double* W; const double* kf; int nops;     // fill pass: stencil weights, folded known-F weights
    void* rowptr; void* col; double* values;         // outputs, int32 or int64 indices; values [nops][nnz]
    long long nnz;
};

// interpolation operators (wlsqm_operator.cu): per query q, the coefficient rows c_q = (Taylor terms at x[q] - xi[I[q]])
// applied to coef, contracted with the block of case I[q].  The queries are sorted stably by I; one warp per run of
// equal I reads that case's block once.  Runs of index nmodels hold the queries whose I is outside [0, nmodels).
struct InterpRuns {
    int* keys; int* keys_sorted;                     // [nx] clamped I, sorted
    int* qidx; int* perm;                            // [nx] 0..nx-1, and the query of each sorted position
    int* run_case; int* run_len; int* run_off;       // [nx] per run (the first *nruns are valid)
    int* nruns;                                      // [1]
};
struct InterpStencilParams {
    const CaseMeta* meta;
    CaseMeta uni;
    int geom_uniform;
    long long op_stride;
    long long nmodels;
    const double* op;
    const double* xi;                                // [nmodels][dim] model origins
    const double* x; long long x_s0;                 // queries
    int dim;
    long long nx;
    const int* run_case; const int* run_len; const int* run_off; const int* nruns; const int* perm;
    const double* coef;                              // [nops][maxno]
    int nops, maxnk, maxno;
    int opc;                                         // operators formed per pass over a query (per-warp shared space)
    double* W;                                       // [nops][nx][maxnk]
    double* K;                                       // [nops][nx][maxno] or nullptr
    double* kf;                                      // [nops][nx] known-F weight for centre folding, or nullptr
    int stages, stage_doubles, ring_off, cq_off, cq_doubles, bar_off_bytes;
    // continuous mode: the rows are the (query, model) pairs (nx of them, I = J), row p is evaluated at query
    // row_query[p] and its coefficient rows are scaled by row_scale[p]; nullptr in nearest mode
    const int* row_query;
    const double* row_scale;
};

// continuous-mode interpolation operators (wlsqm_operator.cu): per query the pairs (q, m) of the models within r, in
// ascending m (pair_ptr [nx + 1], J [npairs] from the ball search over the model grid); per pair the normalised weight
// alpha and its query.  The CSR rows merge the candidates of each query's pairs: L = maxnk + 1 slots per pair
// (neighbours k < nk_m, then the folded known F), slot order = candidate order.  Rows of at most row_cap slots are
// sorted by one warp in shared memory (cont_row_kernel); longer rows by cub's segmented sort over chunks of queries.
constexpr int CONT_ROW_WARPS = 8;
constexpr unsigned CONT_NO_COLUMN = 0xffffffffu;
struct ContCsrParams {
    const CaseMeta* meta;
    CaseMeta uni;
    long long nx, npairs;
    const long long* pair_ptr;                       // [nx + 1]
    const long long* J;                              // [npairs]
    const int* pair_query;                           // [npairs]
    const int32_t* hoods; int hoods_s0;
    long long center;
    int L;                                           // maxnk + 1 candidate slots per pair
    int row_cap;                                     // rows of at most row_cap slots: cont_row_kernel (a power of two, or 0)
    long long* cnt;                                  // count: distinct columns of each row [nx + 1]
    const long long* rp;                             // fill: exclusive scan of cnt
    // sort route, one chunk: queries [q0, q1), slots [slot0, slot0 + nslots)
    long long q0, q1, slot0, nslots;
    int* seg;                                        // [q1 - q0 + 1] first chunk slot of each query
    unsigned* keys; int* cand;                       // [nslots] column (or CONT_NO_COLUMN), chunk slot
    const unsigned* keys_sorted; const int* cand_sorted;
    int* head;                                       // [nslots + 1]: 1 at the first slot of each (query, column) run
    const int* hpos;                                 // exclusive scan of head
    const double* W; const double* kf; int nops, maxnk;
    void* rowptr; void* col; double* values;
    long long nnz;
};

#ifdef __CUDACC__
// Record of case c.  UNI: every case has the sizes of `uni` (only the knowns pattern may vary per case, read from meta
// when given) and the blocks are op_stride apart; otherwise the per-case record.
template <bool UNI>
__device__ __forceinline__ CaseMeta case_meta(const CaseMeta* meta, const CaseMeta& uni, long long op_stride, long long c) {
    CaseMeta m;
    if (UNI) {
        m = uni;
        m.op_off = c * op_stride;
        if (meta) m.knowns = meta[c].knowns;
    } else {
        m = meta[c];
    }
    return m;
}
// bytes of a case's operator block as one bulk copy (a multiple of 16; blocks start 16 B aligned)
__device__ __forceinline__ uint32_t op_block_bytes(const CaseMeta& m) {
    return ((uint32_t)((m.nk + m.nkn) * (int)m.nr) * 8u + 15u) & ~15u;
}

// One warp's ring of S shared-memory stages, filled by 1D bulk copies that complete on one mbarrier per stage.  The
// units [lo, end) are dealt to the warps of the grid in turn; this warp takes first, first + stride, ... (n_my of them).
// Lane 0 keeps the next S - 1 units in flight while the warp works on the current one.  Per unit i (unit u):
//   refill(lane, i, u, issue)   lane 0 starts unit u + (S - 1) * stride in the stage that release() freed last (S == 1:
//                               the current stage, nothing is in flight ahead)
//   wait()                      before the first read of the stage (cur())
//   release()                   after the last read: every lane is done with the stage before lane 0 re-arms it
// issue(stage address, barrier address, unit) is the kernel's: it arms the barrier with the unit's byte count and starts
// the copies; it is taken by reference (passed by value, it changed solve_pack_fields_kernel<1>'s register allocation and
// cost it 5 % of its time on a B200).  Every lane must call start() before the loop.
struct WarpRing {
    uint32_t base, bars, stage_bytes;
    int S, stage = 0;
    uint32_t phase = 0;
    long long first, stride, n_my;

    __device__ __forceinline__ WarpRing(uint32_t base_, uint32_t bars_, int S_, uint32_t stage_bytes_, long long lo,
                                        long long end)
        : base(base_), bars(bars_), stage_bytes(stage_bytes_), S(S_) {
        const int nwarps = blockDim.x >> 5;
        first = lo + (long long)blockIdx.x * nwarps + (threadIdx.x >> 5);
        stride = (long long)gridDim.x * nwarps;
        n_my = first < end ? (end - first + stride - 1) / stride : 0;
    }
    __device__ __forceinline__ uint32_t addr(int s) const { return base + (uint32_t)s * stage_bytes; }
    __device__ __forceinline__ uint32_t bar(int s) const { return bars + (uint32_t)s * 8u; }
    __device__ __forceinline__ uint32_t cur() const { return addr(stage); }
    template <class Issue>
    __device__ __forceinline__ void start(int lane, const Issue& issue) {
        if (lane == 0) {
            for (int s = 0; s < S; ++s) mbar_init_u32(bar(s), 1);
            fence_mbar_init();
            for (int s = 0; s < S - 1 && s < n_my; ++s) issue(addr(s), bar(s), first + (long long)s * stride);
        }
        __syncwarp();
    }
    template <class Issue>
    __device__ __forceinline__ void refill(int lane, long long i, long long unit, const Issue& issue) {
        if (lane == 0 && i + S - 1 < n_my) {
            int sn = stage + S - 1;
            if (sn >= S) sn -= S;
            issue(addr(sn), bar(sn), unit + (long long)(S - 1) * stride);
        }
    }
    __device__ __forceinline__ void wait() const { mbar_wait_u32(bar(stage), phase); }
    __device__ __forceinline__ void release() {
        __syncwarp();
        if (++stage == S) { stage = 0; phase ^= 1u; }
    }
};
#endif

struct InterpParams {
    int dim;
    long long nx;
    const double* x; long long x_s0;                 // [nx][dim]
    const long long* I;                              // [nx] model index, or nullptr (single model 0)
    long long nmodels;                               // indices outside [0, nmodels) give NaN (0: not checked)
    const double* xi; long long xi_s0;               // model origins [nmodels][dim]
    const double* fi; long long fi_s0;               // model coefficients [nmodels][fi_s0]
    const signed char* order; int order_uniform;     // per-model order, or uniform
    int diff;                                        // DOF slot to differentiate to, or -1: all slots
    double* out; long long out_s0;                   // [nx] (diff >= 0) or [nx][out_s0]
    int stage_no;                                    // all slots, every model has stage_no DOFs and out_s0 == stage_no:
                                                     // results are transposed through shared memory (else 0)
};

// Several fields per launch (wlsqm_interp_fields.cu): P.fi / P.out point at the first field of the pass, field j at
// + j * fi_sf / + j * out_sf; P.out_s0 is the query stride of out in both modes.
struct InterpFieldsParams {
    InterpParams P;
    long long fi_sf, out_sf;
    int nf;                                          // fields of this pass (<= 8)
    int width;                                       // all slots: slots written per query (max no), zeros beyond no_i
};

// thread-local message behind wlsqm_last_error() (wlsqm_capi.cu)
void set_last_error(const char* msg);

cudaError_t launch_prepare_smem(int dim, const PrepareParams& P, int blocks, int threads, size_t smem, cudaStream_t st);
int prep_reg_fit_doubles(int dim, int maxorder, int nb, int nkn_max);
int prep_reg_warp_doubles(int dim, int maxorder, int nb, int nkn_max);
int prep_reg_fits_per_warp(int dim, int maxorder);
int prep_reg_max_threads(int dim, int order);
cudaError_t prepare_reg_occupancy(int dim, int maxorder, int threads, size_t smem, int* ctas_per_sm, bool direct = false);
bool prepare_reg_direct_ok(int dim, int maxorder);
cudaError_t launch_prepare_reg(int dim, int maxorder, const PrepRegParams& P, int blocks, int threads, size_t smem,
                               cudaStream_t st);
cudaError_t launch_solve(int dim, const SolveParams& P, int blocks, int threads, size_t smem, cudaStream_t st);
cudaError_t launch_solve_pack(const SolveParams& P, int blocks, int threads, size_t smem, cudaStream_t st);
cudaError_t launch_solve_fields(int dim, const FieldsParams& F, int blocks, int threads, size_t smem, cudaStream_t st);
cudaError_t launch_solve_pack_fields(const FieldsParams& F, int blocks, int threads, size_t smem, cudaStream_t st);
cudaError_t launch_scatter_fi(const CaseMeta* meta, const CaseMeta& uni, long long ncases, const double* fi_case,
                              int fi_case_ld, double* fi_out, long long fi_out_s0, cudaStream_t st);
cudaError_t launch_interpolate(const InterpParams& P, cudaStream_t st);
cudaError_t launch_stencils(const StencilParams& P, int blocks, int threads, size_t smem, cudaStream_t st);
cudaError_t launch_csr_count(const CsrParams& P, cudaStream_t st);
cudaError_t csr_scan(long long* cnt, long long* rp, long long n1, void* tmp, size_t* tmp_bytes, cudaStream_t st);
cudaError_t launch_csr_fill(const CsrParams& P, int index_bits, cudaStream_t st);
cudaError_t interp_runs(const long long* I, long long nx, long long nmodels, const InterpRuns& R, void* tmp, size_t* tmp_bytes,
                        cudaStream_t st);
cudaError_t launch_interp_stencils(const InterpStencilParams& P, int blocks, int threads, size_t smem, cudaStream_t st);
cudaError_t launch_cont_weights(const double* x, long long x_s0, int dim, const double* xi, long long nx, double r,
                                const long long* pair_ptr, const int32_t* J32, long long* J, int* pair_query, double* alpha,
                                cudaStream_t st);
cudaError_t launch_ptr_mismatch(const long long* a, const long long* b, long long n, int* flag, cudaStream_t st);
cudaError_t launch_cont_rows(const ContCsrParams& P, bool fill, int index_bits, cudaStream_t st);
cudaError_t cont_long_rows(const ContCsrParams& P, bool fill, int index_bits, void* tmp, size_t* tmp_bytes, cudaStream_t st);
struct GridView;
cudaError_t launch_interpolate_continuous(const InterpParams& P, const GridView& g, double r, cudaStream_t st);
int interp_fields_per_pass(long long nf, long long ncases, int maxno, long long nx, double rows_per_query,
                           double query_bytes, double out_bytes, long long l2_bytes);
cudaError_t launch_interpolate_fields(const InterpFieldsParams& F, cudaStream_t st);
cudaError_t launch_compact_rows(const double* src, long long sf, long long s0, int nfp, long long n, int maxno, double* dst,
                                cudaStream_t st);
cudaError_t launch_interpolate_continuous_fields(const InterpFieldsParams& F, const GridView& g, double r, cudaStream_t st);
cudaError_t launch_getrf(int n, long long nlhs, double* A, int* ipiv, cudaStream_t st);
cudaError_t launch_getrs(int n, long long nlhs, const double* LU, const int* ipiv, double* b, cudaStream_t st);
cudaError_t launch_gesv(int n, long long nlhs, double* A, int* ipiv, double* b, cudaStream_t st);
cudaError_t launch_sy(int n, long long nlhs, double* A, int* ipiv, double* b, int do_factor, cudaStream_t st);
cudaError_t launch_symmetrize(int n, long long nlhs, double* A, cudaStream_t st);
cudaError_t launch_gtsv(int n, double* dl, double* d, double* du, double* b, cudaStream_t st);
cudaError_t launch_rescale(int nrows, int ncols, long long nlhs, double* A, int algo, double* row_scale, double* col_scale,
                           int* ok, cudaStream_t st);
cudaError_t launch_cond(int n_max, long long ncases, const CaseMeta* meta, const CaseMeta& uni, const double* As,
                        int as_stride, double* cond, cudaStream_t st);

}  // namespace wlsqm
