// wlsqm_capi.cu -- the C ABI declared in include/wlsqm_b200.h: solver handle, device state, staging of
// host arrays, launch configuration.  No numerics live here; see wlsqm_prepare.cu / wlsqm_solve.cu /
// wlsqm_interp.cu / wlsqm_lapack.cu.  There is deliberately no CPU code path: every compute entry
// point needs a CUDA device and fails with WLSQM_E_CUDA otherwise.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "../../include/wlsqm_b200.h"
#include "wlsqm_common.cuh"
#include "wlsqm_kernels.h"
#include "wlsqm_grid.h"
#include "wlsqm_mem.h"
#include "wlsqm_host.h"

namespace wlsqm {
GridView grid_view(const wlsqm_grid* g);
}

using namespace wlsqm;

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

}  // namespace
namespace wlsqm {
void set_last_error(const char* msg) { g_err = msg ? msg : ""; }
}  // namespace wlsqm
namespace {

#define CU(expr)                                                                                   \
    do {                                                                                           \
        cudaError_t e__ = (expr);                                                                  \
        if (e__ != cudaSuccess)                                                                    \
            return fail(e__ == cudaErrorMemoryAllocation ? WLSQM_E_MEMORY : WLSQM_E_CUDA, "%s: %s", #expr, \
                        cudaGetErrorString(e__));                                                  \
    } while (0)

constexpr size_t SMEM_PER_SM = 228 * 1024;      // B200: 228 KB per SM, 227 KB per CTA, 1 KB reserved per CTA
constexpr size_t SMEM_PER_CTA = 227 * 1024;

inline int even(int v) { return (v + 1) & ~1; }

int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}

// One look at the four metadata arrays of a batch (20 bytes per case): which of them hold one value throughout, and --
// only for those that do not -- the reductions the callers need.  The pass is bound by host memory bandwidth (about
// 1 ms per million cases on one thread), so large batches are split over the library's host threads.
struct MetaScan {
    bool same_nk = true, same_order = true, same_knowns = true, same_wm = true;
    int32_t max_nk = 0, min_order = 0, max_order = 0;
    bool uniform() const { return same_nk && same_order && same_knowns && same_wm; }
};
MetaScan scan_meta(long long n, const int32_t* nk, const int32_t* order, const int64_t* knowns, const int32_t* wm) {
    MetaScan r;
    if (n < 1) return r;
    r.max_nk = nk[0]; r.min_order = r.max_order = order[0];
    if (n < 2) return r;
    const int32_t nk0 = nk[0], od0 = order[0], wm0 = wm[0];
    const int64_t kn0 = knowns[0];
    std::atomic<uint32_t> d_nk{0}, d_od{0}, d_wm{0};
    std::atomic<uint64_t> d_kn{0};
    auto piece = [&](size_t lo, size_t hi) {
        uint32_t a = 0, b = 0, c = 0;
        uint64_t d = 0;
        for (size_t i = lo; i < hi; ++i) a |= (uint32_t)(nk[i] ^ nk0);
        for (size_t i = lo; i < hi; ++i) b |= (uint32_t)(order[i] ^ od0);
        for (size_t i = lo; i < hi; ++i) c |= (uint32_t)(wm[i] ^ wm0);
        for (size_t i = lo; i < hi; ++i) d |= (uint64_t)(knowns[i] ^ kn0);
        if (a) d_nk.fetch_or(a, std::memory_order_relaxed);
        if (b) d_od.fetch_or(b, std::memory_order_relaxed);
        if (c) d_wm.fetch_or(c, std::memory_order_relaxed);
        if (d) d_kn.fetch_or(d, std::memory_order_relaxed);
    };
    const bool par = n >= 262144 && env_int("WLSQM_META_THREADS", 1) != 0;
    if (par) par_for((size_t)n, piece);
    else piece(0, (size_t)n);
    r.same_nk = d_nk.load() == 0; r.same_order = d_od.load() == 0; r.same_wm = d_wm.load() == 0; r.same_knowns = d_kn.load() == 0;
    if (!r.same_nk || !r.same_order) {
        std::atomic<int32_t> mk{nk0}, lo_o{od0}, hi_o{od0};
        auto atomic_max = [](std::atomic<int32_t>& t, int32_t v) { int32_t c = t.load(); while (v > c && !t.compare_exchange_weak(c, v)) {} };
        auto atomic_min = [](std::atomic<int32_t>& t, int32_t v) { int32_t c = t.load(); while (v < c && !t.compare_exchange_weak(c, v)) {} };
        auto red = [&](size_t lo, size_t hi) {
            int32_t m = nk0, l = od0, h = od0;
            if (!r.same_nk)
                for (size_t i = lo; i < hi; ++i) m = nk[i] > m ? nk[i] : m;
            if (!r.same_order)
                for (size_t i = lo; i < hi; ++i) { l = order[i] < l ? order[i] : l; h = order[i] > h ? order[i] : h; }
            atomic_max(mk, m); atomic_min(lo_o, l); atomic_max(hi_o, h);
        };
        if (par) par_for((size_t)n, red);
        else red(0, (size_t)n);
        r.max_nk = mk.load(); r.min_order = lo_o.load(); r.max_order = hi_o.load();
    }
    return r;
}

// 1 = device-accessible (device or managed), 0 = host (pinned or pageable)
int is_device_ptr(const void* p) {
    if (!p) return 0;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// A device buffer that only grows.  Blocks come from the library's memory pool (wlsqm_mem.h).
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return WLSQM_OK;
        if (p) dev_free_sync(p);     // growing a live buffer: earlier work may still read the old block
        p = nullptr;
        cap = 0;
        if (bytes == 0) return WLSQM_OK;
        cudaError_t e = dev_alloc(&p, bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(WLSQM_E_MEMORY, "device allocation of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
        }
        cap = bytes;
        return WLSQM_OK;
    }
    // the caller has synchronised the streams that used the buffer
    void release() {
        if (p) dev_free(p);
        p = nullptr;
        cap = 0;
    }
};

// dst[f][i][k][0..w) = src[f][idx[i][k]][0..w) for the nf fields f (src field stride src_sf, dst field stride dst_sf).
// Only the first nk_i neighbours of case i are read (nk_i from the per-case records, else nk_uni; negative: all k
// columns): the padding of a ragged hood array (cKDTree and wlsqm_grid_knn both report missing neighbours as the index
// n) is never dereferenced and its slots are zero-filled.  An index outside [0, nsrc) among the USED slots -- where the
// reference's x[hoods] raises IndexError -- gives NaN and raises *err.
__global__ void gather_hoods_kernel(const double* __restrict__ src, long long src_s0, int w, const int32_t* __restrict__ idx,
                                    long long idx_s0, long long n, int k, double* __restrict__ dst, long long nsrc,
                                    const CaseMeta* __restrict__ meta, int nk_uni, int* __restrict__ err, int nf = 1,
                                    long long src_sf = 0, long long dst_sf = 0) {
    const long long per = (long long)k * w;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n * per;
         t += (long long)gridDim.x * blockDim.x) {
        const long long i = t / per;
        const int r = (int)(t - i * per);
        const int kk = r / w, d = r - kk * w;
        const int nki = meta ? meta[i].nk : (nk_uni >= 0 ? nk_uni : k);
        if (kk < nki) {
            const long long j = idx[i * idx_s0 + kk];
            if (j >= 0 && j < nsrc) {
                for (int f = 0; f < nf; ++f) dst[t + f * dst_sf] = src[f * src_sf + j * src_s0 + d];
            } else {
                for (int f = 0; f < nf; ++f) dst[t + f * dst_sf] = __longlong_as_double(0x7ff8000000000000LL);
                if (err) *err = 1;
            }
        } else {
            for (int f = 0; f < nf; ++f) dst[t + f * dst_sf] = 0.0;
        }
    }
}

// strided 3-level copy  dst[i][a][b] <- src[i*s0 + a*s1 + b*s2], dst dense
__global__ void gather3_kernel(double* __restrict__ dst, const double* __restrict__ src, long long n, int na, int nb,
                               long long s0, long long s1, long long s2) {
    const long long per = (long long)na * nb;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n * per;
         t += (long long)gridDim.x * blockDim.x) {
        const long long i = t / per;
        const int r = (int)(t - i * per);
        const int a = r / nb, b = r - a * nb;
        dst[t] = src[i * s0 + a * s1 + b * s2];
    }
}

}  // namespace

struct wlsqm_solver {
    int dim = 0, device = 0, algorithm = 1, do_sens = 0, max_iter = 0, debug = 0;
    long long ncases = 0;
    int maxnk = 0, maxno = 1, maxnr = 0, maxnq = 0, maxorder = 0, maxnkn = 0;
    bool uniform = true, any_knowns = false, uniform_no = true;
    bool last_nk_odd = false;   // nk of the LAST case is odd (see the bulk copies of fk rows in wlsqm_solver_solve)
    bool geom_uniform = true;   // same nk / order / weighting / number of knowns everywhere (the knowns pattern may vary)
    CaseMeta uni{};
    long long op_stride = 0, op_total = 0;
    std::vector<CaseMeta> hmeta;
    CaseMeta* dmeta = nullptr;
    signed char* dorder = nullptr;
    double* op = nullptr;
    double* fi_case = nullptr;
    // wlsqm_solver_keep_solution(s, 0): solve() with a device fi writes the caller's array only; interpolate() needs the copy
    bool keep_solution = true, fi_case_valid = true;
    int l2_bytes = 0;                            // L2 size of the device (interpolate_fields' pass plan)
    double* xi_dev = nullptr;
    double* As = nullptr;
    int as_stride = 0;
    int* iters_dev = nullptr;   // [0] = max, [1..ncases] per case (ITERATIVE only)
    bool ready = false;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t s_in = nullptr, s_out = nullptr;   // H2D / D2H streams of the staged (host-pointer) pipeline
    std::vector<cudaEvent_t> events;
    int sm_count = 148;
    DevBuf xk_keep;             // dense copy of xk (ALGO_ITERATIVE needs the geometry at solve time)
    DevBuf st_xk, st_fk, st_fi, st_sens, st_x, st_I, st_out;
    DevBuf hoods_dev, hood_x, hood_f, hood_fk;   // prepare_hoods / solve_hoods: neighbour lists and gathered data
    long long hood_points = 0;
    bool hoods_current = false;                  // the LAST prepare was prepare_hoods: hoods_dev belongs to the operators
    DevBuf opx_coef;                             // operator export: device copy of the coefficient rows
    DevBuf opx_runs, opx_tmp;                    // interpolation operators: runs of the sorted queries, cub scratch
    int* hood_err = nullptr;                     // device flag: a used hood index fell outside [0, npoints)
    // fused result gather: global solution arrays of the GPUs of the job (peer memory), see wlsqm_solver_set_gather
    int ngather = 0;
    double* gather[WLSQM_MAX_PEERS] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    long long gather_row0 = 0, gather_s0 = 0;
    wlsqm_grid* models_grid = nullptr;           // search grid over the model origins (index_models)
    wlsqm_solver* lender = nullptr;              // guest mode: op / dmeta / dorder / xi_dev / As / xk_keep belong to this solver
    long long bytes_state = 0;
    // batches of mixed orders: case lists per order (device, ascending case index inside an order), so that prepare()
    // runs one kernel instantiation per order instead of the maximum order's for every case
    int* order_perm = nullptr;
    long long order_lo[6] = {0, 0, 0, 0, 0, 0};
};

namespace {

long long staging_bytes(const wlsqm_solver* s) {
    return (long long)(s->xk_keep.cap + s->st_xk.cap + s->st_fk.cap + s->st_fi.cap + s->st_sens.cap + s->st_x.cap +
                       s->st_I.cap + s->st_out.cap + s->hoods_dev.cap + s->hood_x.cap + s->hood_f.cap + s->hood_fk.cap +
                       s->opx_coef.cap + s->opx_runs.cap + s->opx_tmp.cap);
}

int use_device(const wlsqm_solver* s) {
    CU(cudaSetDevice(s->device));
    return WLSQM_OK;
}

// dst[f][i][0..k*w) = the first nk_i neighbours of case i in the solver's neighbour lists (prepare_hoods), w values each,
// from src[f] (points of the last prepare_hoods), for the nf fields f; on the solver's stream
cudaError_t gather_hoods(const wlsqm_solver* s, const double* src, long long src_s0, int w, int k, double* dst, int* err,
                         int nf = 1, long long src_sf = 0, long long dst_sf = 0) {
    const long long total = s->ncases * k * w;
    gather_hoods_kernel<<<(unsigned)std::min<long long>((total + 255) / 256, (long long)s->sm_count * 32), 256, 0, s->stream>>>(
        src, src_s0, w, (const int32_t*)s->hoods_dev.p, s->maxnk, s->ncases, k, dst, s->hood_points, s->dmeta, s->uni.nk, err,
        nf, src_sf, dst_sf);
    return cudaGetLastError();
}

// the fields of a solve launch that come from the solver: records, operators, algorithm, the geometry the refinement
// reads, and (ALGO_ITERATIVE) its iteration counters, which the caller clears
void solve_params(const wlsqm_solver* s, SolveParams& P) {
    P.meta = s->dmeta; P.uni = s->uni; P.op_stride = s->op_stride; P.ncases = s->ncases; P.op = s->op;
    P.geom_uniform = s->geom_uniform ? 1 : 0;
    P.algorithm = s->algorithm; P.max_iter = s->max_iter;
    P.xi = s->xi_dev; P.xi_s0 = s->dim;
    P.xk = (const double*)s->xk_keep.p; P.xk_s0 = (long long)s->maxnk * s->dim; P.xk_s1 = s->dim;
    if (s->algorithm == WLSQM_ALGO_ITERATIVE) {
        P.iters_max = s->iters_dev;
        P.iters_case = s->iters_dev + 1;
    }
}

// One solve launch over the cases [P.case_lo, P.ncases): config(rows) sets the launch shape for `rows` cases, launch()
// starts the kernel.  Rows of fk with an odd element count are fetched by bulk copies of one element more (inside the
// even row pitch, wlsqm_solve.cu), but the storage of a caller's strided device array may end with the last element of
// its last row: with `odd_last` (the launch ends with the last case, whose nk is odd) and bulk copies of fk, that one
// case runs in a launch of its own with plain loads.
template <class Config, class Launch>
int launch_solve_split(SolveParams& P, bool odd_last, Config config, Launch launch) {
    const long long c0 = P.case_lo, c1 = P.ncases;
    int rc = config(c1 - c0);
    if (rc) return rc;
    if (odd_last && P.f_tma) {
        if (c1 - c0 > 1) {
            P.ncases = c1 - 1;
            rc = config(c1 - c0 - 1);
            if (rc) return rc;
            CU(launch());
        }
        P.case_lo = c1 - 1;
        P.ncases = c1;
        rc = config(1);
        if (rc) return rc;
        P.f_tma = 0;
    }
    CU(launch());
    return WLSQM_OK;
}

// ---- launch configuration ------------------------------------------------------------------------
struct LaunchCfg { int blocks, threads; size_t smem; };

// Grid of a kernel whose CTAs of `warps` warps and `smem` bytes each take units in turn: as many CTAs per SM as shared
// memory holds (1 KB of it reserved per CTA), at most max_warps_sm / warps of them (at least one), and no more CTAs
// than the units fill.
int grid_blocks(const wlsqm_solver* s, size_t smem, int warps, int max_warps_sm, long long units) {
    int ctas = (int)(SMEM_PER_SM / (smem + 1024));
    ctas = std::max(1, std::min(ctas, std::max(1, max_warps_sm / warps)));
    const long long need = (units + warps - 1) / warps;
    return (int)std::max<long long>(1, std::min<long long>((long long)s->sm_count * ctas, need));
}

int config_prepare(const wlsqm_solver* s, PrepareParams& P, LaunchCfg& L) {
    const int nk = std::max(s->maxnk, 1), no = s->maxno, nr = std::max(s->maxnr, 1), nq = std::max(s->maxnq, 1);
    const int cs = no | 1, lda = nr | 1, sq = nq | 1;
    int off = 0;
    off += even(nk * cs);       P.off_w = off;
    off += even(nk);            P.off_a = off;
    off += even(nr * lda);      P.off_rs = off;
    off += even(nr);            P.off_s = off;
    off += even(nr * sq);       P.off_i = off;
    off += 36;
    P.warp_doubles = off;
    const size_t per_warp = (size_t)off * 8;
    if (per_warp > SMEM_PER_CTA)
        return fail(WLSQM_E_VALUE, "case too large for shared memory (nk=%d, no=%d): %zu bytes per fit", nk, no, per_warp);
    int warps = env_int("WLSQM_PREP_WARPS", 8);
    warps = std::max(1, std::min(warps, PREP_MAX_THREADS / 32));
    while (warps > 1 && warps * per_warp > SMEM_PER_CTA) --warps;
    L.threads = warps * 32;
    L.smem = warps * per_warp;
    L.blocks = grid_blocks(s, L.smem, warps, 48, s->ncases);
    return WLSQM_OK;
}

// register/DMMA kernel: false if the fit does not fit its shared-memory carve-up (then the smem kernel runs)
// (order_sel / count: the launch covers `count` cases of order `order_sel` only -- batches of mixed orders)
bool config_prepare_reg(const wlsqm_solver* s, PrepRegParams& P, LaunchCfg& L, bool direct = false, int order_sel = -1,
                        long long count = -1) {
    const int kord = order_sel >= 0 ? order_sel : s->maxorder;
    const long long ncases = count >= 0 ? count : s->ncases;
    const int nkp = (std::max(s->maxnk, 1) + 3) & ~3;
    P.nb = (std::max(nkp, s->maxnq) + 31) / 32;
    const int nkn_max = s->maxnq > 0 ? s->maxnkn : 0;
    P.fit_doubles = prep_reg_fit_doubles(s->dim, kord, P.nb, nkn_max);
    P.warp_doubles = prep_reg_warp_doubles(s->dim, kord, P.nb, nkn_max);
    const int fpw = prep_reg_fits_per_warp(s->dim, kord);
    const size_t per_warp = (size_t)P.warp_doubles * 8;
    if (per_warp > SMEM_PER_CTA) return false;
    // CTA size: the one that keeps most warps resident (shared memory and registers both limit it).  The answer depends
    // only on (kernel instantiation, bytes per warp): remembered, so that a small one-shot fit does not pay sixteen
    // occupancy queries (tens of microseconds) on every call.
    int best_w = 0, best_ctas = 0;
    const int force_w = env_int("WLSQM_PREP_WARPS", 0);
    struct OccKey { int dim, ord, direct, force; size_t per_warp; int w, ctas; };
    static std::mutex occ_mu;
    static std::vector<OccKey> occ_cache;
    {
        std::lock_guard<std::mutex> lock(occ_mu);
        for (const OccKey& k : occ_cache)
            if (k.dim == s->dim && k.ord == kord && k.direct == (int)direct && k.force == force_w && k.per_warp == per_warp) {
                best_w = k.w; best_ctas = k.ctas;
                break;
            }
    }
    const bool cached = best_w > 0;
    // (whole multiples of the four schedulers first -- 18 warps measured slower than 16 for 3D order 3 -- then any size)
    for (int pass = 0; !cached && pass < 2 && best_w < 1; ++pass)
    for (int w = 1; w <= prep_reg_max_threads(s->dim, kord) / 32; ++w) {
        if (force_w > 0 && w != force_w) continue;
        if (pass == 0 && force_w <= 0 && (w & 3)) continue;
        if (w * per_warp > SMEM_PER_CTA) break;
        int c = 0;
        if (prepare_reg_occupancy(s->dim, kord, w * 32, w * per_warp, &c, direct) != cudaSuccess) {
            cudaGetLastError();
            continue;
        }
        // among the CTA sizes that keep the most warps resident, the LARGEST: the warps of one CTA start together and
        // stay roughly in phase, so they share instruction-cache lines of this kernel's ~75 KB of straight-line code
        // (measured, 2D order 4: one 16-warp CTA per SM 4.71 ms, four 4-warp CTAs 5.26 ms)
        if (w * c >= best_w * best_ctas) { best_w = w; best_ctas = c; }
    }
    if (best_w < 1 || best_ctas < 1) return false;
    if (!cached) {
        std::lock_guard<std::mutex> lock(occ_mu);
        occ_cache.push_back(OccKey{s->dim, kord, (int)direct, force_w, per_warp, best_w, best_ctas});
    }
    const int warps = best_w;
    int ctas = best_ctas;
    L.threads = warps * 32;
    L.smem = warps * per_warp;
    P.phase_sync = env_int("WLSQM_PREP_PHASE_SYNC", 0);
    const int cap = env_int("WLSQM_PREP_CTAS", 0);
    if (cap > 0) ctas = std::min(ctas, cap);
    long long need = (ncases + (long long)warps * fpw - 1) / ((long long)warps * fpw);
    L.blocks = (int)std::max<long long>(1, std::min<long long>((long long)s->sm_count * ctas, need));
    return true;
}

int config_solve(const wlsqm_solver* s, SolveParams& P, LaunchCfg& L, long long ncases_launch) {
    const bool iter = s->algorithm == WLSQM_ALGO_ITERATIVE;
    // one stage of the per-warp ring: [operator block | fext = fk + known fi | xk (ALGO_ITERATIVE)]
    const int op_doubles = std::max(2, even(s->maxnq * s->maxnr));
    const int f_doubles = std::max(2, even(s->maxnq));
    const int x_doubles = iter ? std::max(2, even(s->maxnk * s->dim)) : 0;
    const int stage_doubles = op_doubles + f_doubles + x_doubles;
    const size_t stage_bytes = (size_t)stage_doubles * 8;
    // Measured on B200 (profiles/README.md): a ring of 2 stages and ONE CTA per SM with as many warps as
    // fit (16 for the headline block size) streams best; deeper rings or several CTAs per SM put more
    // distant operator blocks in flight at once and lose HBM efficiency.  Blocks under 3 KB are bound by
    // per-case issue overhead instead and want two such CTAs per SM.
    // ALGO_ITERATIVE keeps a warp busy on one block for thousands of cycles: more resident warps (one stage
    // each) beat prefetch depth there (measured: 3D order 4 k=60 with sens, 16.7 -> 9.6 ms per 1M points).
    // Batches whose cases differ in size (ALGO_BASIC): when two stages of the LARGEST block leave room for fewer than
    // 16 warps, one stage and twice the warps win -- the typical block is smaller than the stage, so resident warps put
    // more bytes in flight than a prefetch slot sized for the worst case (measured, 400k cases 3D orders 2-4 nk 40-60:
    // 2 stages x 6 warps 1.21 ms, 1 stage x 12 warps 0.73 ms = 0.78 of the HBM peak)
    const bool hetero_shallow = !iter && !s->geom_uniform && 16 * (2 * stage_bytes + 512) > SMEM_PER_CTA;
    int S = env_int("WLSQM_SOLVE_STAGES", ((iter && stage_bytes >= 8192) || hetero_shallow) ? 1 : 2);
    S = std::max(1, std::min(S, 8));
    // ALGO_ITERATIVE in 1D / 2D: one 24-warp CTA per SM at 80 registers (the refinement loop is latency-bound: 24 resident
    // warps beat 16, and one CTA whose warps start together beats two 12-warp CTAs: 1.59 -> 1.54 ms)
    const bool iter_small = iter && s->dim < 3;
    const int max_warps = (iter ? (iter_small ? SOLVE_ITER12_THREADS : SOLVE_MAX_THREADS_ITER) : SOLVE_MAX_THREADS) / 32;
    // Batches whose cases differ in size: the ring is sized for the largest block but the typical block is smaller, so the
    // pass is bound by per-case issue overhead and bytes in flight like any small-block batch -- as many resident warps as
    // shared memory holds (measured, 1M cases 2D orders 2-4 nk 22-30: 16 warps 0.770 ms, 24 warps 0.589 ms)
    const size_t mean_block_bytes = s->ncases > 0 ? (size_t)(s->op_total * 8 / s->ncases) : stage_bytes;
    const bool small_mean = !iter && !s->geom_uniform && (mean_block_bytes < 3072 || hetero_shallow);
    int warps = env_int("WLSQM_SOLVE_WARPS", iter_small ? 24 : (small_mean ? 32 : 16));
    warps = std::max(1, std::min(warps, max_warps));
    size_t per_warp = 0;
    int off_fi, off_r, wd;
    for (;;) {
        off_fi = S * stage_doubles;
        off_r = off_fi + 36;
        wd = off_r + (iter ? std::max(2, even(s->maxnk)) : 0);
        wd = (wd + 15) & ~15;                      // 128 B granularity per warp slice
        per_warp = (size_t)wd * 8 + (size_t)S * 8;
        if (warps * per_warp <= SMEM_PER_CTA) break;
        if (warps > 4) --warps;
        else if (S > 2) --S;
        else if (warps > 1) --warps;
        else if (S > 1) --S;
        else return fail(WLSQM_E_VALUE, "operator block too large for shared memory (%zu bytes)", stage_bytes);
    }
    P.stages = S;
    P.stage_doubles = stage_doubles;
    P.off_f = op_doubles; P.off_xk = op_doubles + f_doubles;
    P.off_fi = off_fi; P.off_r = off_r;
    P.warp_doubles = wd;
    // bulk-copy eligibility of the data arrays (16 B alignment of every row start, unit stride)
    P.f_tma = (P.fk_s1 == 1 && ((uintptr_t)P.fk % 16 == 0) && (P.fk_s0 % 2 == 0)) ? 1 : 0;
    P.xk_tma = (iter && P.xk_s1 == s->dim && ((uintptr_t)P.xk % 16 == 0) && (P.xk_s0 % 2 == 0)) ? 1 : 0;
    if (env_int("WLSQM_SOLVE_NO_FTMA", 0)) P.f_tma = P.xk_tma = 0;
    P.bar_off_bytes = warps * wd * 8;
    L.threads = warps * 32;
    L.smem = (size_t)P.bar_off_bytes + (size_t)warps * S * 8;
    L.blocks = grid_blocks(s, L.smem, warps,
                           env_int("WLSQM_SOLVE_MAXWARPS_SM", iter_small ? 24 : ((stage_bytes >= 3072 && !small_mean) ? 16 : 32)),
                           ncases_launch);
    return WLSQM_OK;
}

// packed solve (several small cases per warp pass): launch configuration; the stage holds
// [CPW operator blocks | CPW fk rows | CPW x nkn known values]
bool pack_eligible(const wlsqm_solver* s) {
    // blocks of 3 KB and more already stream at the HBM roofline with one case per warp (measured)
    return s->geom_uniform && s->algorithm != WLSQM_ALGO_ITERATIVE && s->maxno <= 16 && s->uni.nr > 0 &&
           s->op_stride * 8 < env_int("WLSQM_SOLVE_PACK_BELOW", 3072) && !env_int("WLSQM_SOLVE_NOPACK", 0);
}
int config_solve_pack(const wlsqm_solver* s, SolveParams& P, LaunchCfg& L, long long ncases_launch) {
    const int no = s->uni.no, nk = s->uni.nk, nkn = s->uni.nkn;
    int lw = 0;
    while ((1 << lw) < no) ++lw;
    P.pack_lw = lw;
    const int cpw = 32 >> lw;
    const int op_doubles = cpw * (int)s->op_stride;
    const int f_doubles = std::max(2, even(cpw * nk));
    const int k_doubles = std::max(2, even(cpw * nkn));
    const int stage_doubles = op_doubles + f_doubles + k_doubles;
    const size_t stage_bytes = (size_t)stage_doubles * 8;
    int S = env_int("WLSQM_SOLVE_STAGES", 2);
    S = std::max(2, std::min(S, 8));
    int warps = env_int("WLSQM_SOLVE_WARPS", 32);    // one 32-warp CTA per SM (measured: 0.692 ms against 0.712 ms for 8-warp CTAs, cfg4 2D)
    warps = std::max(1, std::min(warps, SOLVE_MAX_THREADS / 32));
    int wd = 0;
    for (;;) {
        wd = (S * stage_doubles + 15) & ~15;
        if ((size_t)warps * (wd * 8 + S * 8) <= SMEM_PER_CTA) break;
        if (warps > 1) --warps;
        else return fail(WLSQM_E_VALUE, "operator pack too large for shared memory (%zu bytes)", stage_bytes);
    }
    P.stages = S;
    P.stage_doubles = stage_doubles;
    P.off_f = op_doubles; P.off_xk = op_doubles + f_doubles;
    P.warp_doubles = wd;
    // one bulk copy for the CPW fk rows of a pack: dense rows, 16 B aligned pack starts
    P.f_tma = (P.fk_s1 == 1 && P.fk_s0 == nk && ((uintptr_t)P.fk % 16 == 0) && ((cpw * nk) % 2 == 0)) ? 1 : 0;
    if (env_int("WLSQM_SOLVE_NO_FTMA", 0)) P.f_tma = 0;
    P.xk_tma = 0;
    P.bar_off_bytes = warps * wd * 8;
    L.threads = warps * 32;
    L.smem = (size_t)P.bar_off_bytes + (size_t)warps * S * 8;
    L.blocks = grid_blocks(s, L.smem, warps, env_int("WLSQM_SOLVE_MAXWARPS_SM", 32), (ncases_launch + cpw - 1) / cpw);
    return WLSQM_OK;
}

// Field-batched solve: the launch shape of the single-field solve (ring depth, fext / known-value slot sizes, warps per
// CTA -- at most SOLVE_FIELDS_THREADS: 128 registers for the accumulators of 8 fields, or the refinement of a field) with
// every stage widened by one data slot per further field.  F.nf is lowered to the fields that the shared memory of that
// shape holds (at least 1: the single-field shape fits).  F.P.fk / fk strides and F.fk_sf must be set (bulk-copy
// eligibility).
int config_solve_fields(const wlsqm_solver* s, FieldsParams& F, LaunchCfg& L, long long ncases_launch, bool pack) {
    SolveParams& P = F.P;
    const int rc = pack ? config_solve_pack(s, P, L, ncases_launch) : config_solve(s, P, L, ncases_launch);
    if (rc) return rc;
    const bool iter = s->algorithm == WLSQM_ALGO_ITERATIVE;
    const int warps = std::min(L.threads / 32, SOLVE_FIELDS_THREADS / 32);
    const int S = P.stages;
    const int op_d = P.off_f, f_d = P.off_xk - P.off_f, x_d = P.stage_doubles - P.off_xk;
    const int tail = pack ? 0 : 36 + (iter ? std::max(2, even(s->maxnk)) : 0);     // fis + rs per warp (solve_kernel)
    auto stage_of = [&](int nfp) { return pack ? op_d + nfp * (f_d + x_d) : op_d + nfp * f_d + x_d; };
    auto warp_of = [&](int nfp) { return (S * stage_of(nfp) + tail + 15) & ~15; };
    int nfp = std::max(1, F.nf);
    while (nfp > 1 && (size_t)warps * ((size_t)warp_of(nfp) * 8 + (size_t)S * 8) > SMEM_PER_CTA) --nfp;
    F.nf = nfp;
    F.f_doubles = f_d;
    F.k_doubles = pack ? x_d : 0;
    P.stage_doubles = stage_of(nfp);
    P.off_xk = op_d + nfp * f_d;
    P.off_fi = S * P.stage_doubles;
    P.off_r = P.off_fi + 36;
    P.warp_doubles = warp_of(nfp);
    if (nfp > 1 && (F.fk_sf % 2)) P.f_tma = 0;     // every field's rows must start 16 B aligned
    P.bar_off_bytes = warps * P.warp_doubles * 8;
    L.threads = warps * 32;
    L.smem = (size_t)P.bar_off_bytes + (size_t)warps * S * 8;
    const long long units = pack ? (ncases_launch + (32 >> P.pack_lw) - 1) / (32 >> P.pack_lw) : ncases_launch;
    L.blocks = grid_blocks(s, L.smem, warps, 16, units);
    return WLSQM_OK;
}

// copy a pitched host/device 2-D array of doubles into a dense device buffer (rows x width)
int to_dense(double* dst, const double* src, long long rows, long long width, long long pitch, cudaStream_t st) {
    if (rows == 0 || width == 0) return WLSQM_OK;
    if (rows == 1 || pitch == width) {
        CU(cudaMemcpyAsync(dst, src, (size_t)rows * width * 8, cudaMemcpyDefault, st));
        return WLSQM_OK;
    }
    CU(cudaMemcpy2DAsync(dst, (size_t)width * 8, src, (size_t)pitch * 8, (size_t)width * 8, (size_t)rows,
                         cudaMemcpyDefault, st));
    return WLSQM_OK;
}
// below this size the driver's own staging of pageable copies is as fast (measured: 24 MB at 25 GB/s, 240 MB at 12 GB/s)
constexpr long long BOUNCE_MIN_BYTES = 64ll << 20;
// to_dense / from_dense for arrays that may be ordinary pageable host memory: large ones go through the page-locked
// rings with threaded host copies (wlsqm_host.h); the call returns when the host side is done with the array
int stage_in(int device, double* dst, const double* src, long long rows, long long width, long long pitch, cudaStream_t st) {
    if (rows * width * 8 >= BOUNCE_MIN_BYTES && (size_t)width * 8 <= BOUNCE_SLOT_BYTES && env_int("WLSQM_BOUNCE", 1) != 0 &&
        !is_device_ptr(src) && is_pageable_host(src)) {
        bounce_lock();
        const cudaError_t e = h2d_bounced(bounce_rings(device).in, dst, src, rows, width, pitch, st);
        bounce_unlock();
        if (e != cudaSuccess) return fail(WLSQM_E_CUDA, "host -> device staging: %s", cudaGetErrorString(e));
        return WLSQM_OK;
    }
    return to_dense(dst, src, rows, width, pitch, st);
}
int from_dense(double* dst, long long pitch, const double* src, long long src_pitch, long long rows, long long width,
               cudaStream_t st);
int stage_out(int device, double* dst, long long pitch, const double* src, long long src_pitch, long long rows, long long width,
              cudaStream_t st) {
    if (rows * width * 8 >= BOUNCE_MIN_BYTES && (size_t)width * 8 <= BOUNCE_SLOT_BYTES && env_int("WLSQM_BOUNCE", 1) != 0 &&
        !is_device_ptr(dst) && is_pageable_host(dst)) {
        bounce_lock();
        const cudaError_t e = d2h_bounced(bounce_rings(device).out, dst, pitch, src, src_pitch, rows, width, st);
        bounce_unlock();
        if (e != cudaSuccess) return fail(WLSQM_E_CUDA, "device -> host staging: %s", cudaGetErrorString(e));
        return WLSQM_OK;
    }
    return from_dense(dst, pitch, src, src_pitch, rows, width, st);
}
int from_dense(double* dst, long long pitch, const double* src, long long src_pitch, long long rows, long long width,
               cudaStream_t st) {
    if (rows == 0 || width == 0) return WLSQM_OK;
    if (rows == 1 || (pitch == width && src_pitch == width)) {
        CU(cudaMemcpyAsync(dst, src, (size_t)rows * width * 8, cudaMemcpyDefault, st));
        return WLSQM_OK;
    }
    CU(cudaMemcpy2DAsync(dst, (size_t)pitch * 8, src, (size_t)src_pitch * 8, (size_t)width * 8, (size_t)rows,
                         cudaMemcpyDefault, st));
    return WLSQM_OK;
}

bool ranges_overlap(const void* a, long long abytes, const void* b, long long bbytes) {
    const char* a0 = (const char*)a;
    const char* b0 = (const char*)b;
    return a0 < b0 + bbytes && b0 < a0 + abytes;
}

// whether the (field, row, slot) -> element map of an [nf][rows][width] array with element strides sf, s0 and a
// contiguous last axis is injective in one of the two accepted layouts: fields-outer (sf >= (rows-1)*s0 + width,
// s0 >= width) or fields-inner (sf >= width, s0 >= (nf-1)*sf + width).  fitter/fields.py states the same rule.
bool fields_layout_ok(long long nf, long long rows, long long width, long long sf, long long s0) {
    const bool outer = (nf == 1 || sf >= (rows - 1) * s0 + width) && (rows == 1 || s0 >= width);
    const bool inner = (nf == 1 || sf >= width) && (rows == 1 || s0 >= (nf - 1) * sf + width);
    return sf >= 0 && s0 >= 0 && (outer || inner);
}

}  // namespace

extern "C" {

int wlsqm_b200_abi_version(void) { return 1; }
const char* wlsqm_last_error(void) { return g_err.c_str(); }

int wlsqm_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int wlsqm_number_of_dofs(int dimension, int order) { return number_of_dofs(dimension, order); }

void* wlsqm_pinned_alloc(int64_t bytes) {
    void* p = nullptr;
    if (bytes <= 0) return nullptr;
    if (cudaHostAlloc(&p, (size_t)bytes, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
// write-combined page-locked memory: faster for the device to read over PCIe on some hosts, slow for the CPU to read back
// -- for buffers the host only WRITES (the per-step input fk)
void* wlsqm_pinned_alloc_wc(int64_t bytes) {
    void* p = nullptr;
    if (bytes <= 0) return nullptr;
    if (cudaHostAlloc(&p, (size_t)bytes, cudaHostAllocWriteCombined) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
void wlsqm_pinned_free(void* p) {
    if (p) cudaFreeHost(p);
}

// max nk, min / max order and whether every case has the same (nk, order, knowns, weighting), in one vectorised pass
// (the Python mirror needs them for its shape checks; three numpy reductions over 1M cases cost ~1 ms per call)
int wlsqm_meta_summary(int64_t ncases, const int32_t* nk, const int32_t* order, const int64_t* knowns, const int32_t* wm,
                       int32_t* max_nk, int32_t* min_order, int32_t* max_order, int32_t* uniform) {
    if (ncases < 0 || (ncases > 0 && (!nk || !order || !knowns || !wm))) return fail(WLSQM_E_VALUE, "NULL metadata array");
    const MetaScan m = scan_meta(ncases, nk, order, knowns, wm);
    if (max_nk) *max_nk = m.max_nk;
    if (min_order) *min_order = m.min_order;
    if (max_order) *max_order = m.max_order;
    if (uniform) *uniform = m.uniform() ? 1 : 0;
    return WLSQM_OK;
}

int wlsqm_pool_stats(int device, int64_t* reserved, int64_t* used) {
    long long r = -1, u = -1;
    dev_pool_stats(device, &r, &u);
    if (reserved) *reserved = r;
    if (used) *used = u;
    return WLSQM_OK;
}

int wlsqm_pool_trim(int device) {
    if (wlsqm_device_count() < 1) return fail(WLSQM_E_CUDA, "no CUDA device available (there is no CPU fallback)");
    dev_pool_trim(device);
    return WLSQM_OK;
}

int wlsqm_solver_create(int dimension, int64_t ncases, const int32_t* nk, const int32_t* order, const int64_t* knowns,
                        const int32_t* wm, int algorithm, int do_sens, int max_iter, int debug, int device,
                        wlsqm_solver_t** out) {
    if (!out) return fail(WLSQM_E_VALUE, "out is NULL");
    *out = nullptr;
    if (dimension < 1 || dimension > 3) return fail(WLSQM_E_VALUE, "Dimension must be 1, 2 or 3, got %d", dimension);
    if (algorithm != WLSQM_ALGO_BASIC && algorithm != WLSQM_ALGO_ITERATIVE)
        return fail(WLSQM_E_VALUE, "Unknown algorithm specifier %d; see wlsqm.fitter.defs for valid specifiers ALGO_*",
                    algorithm);
    if (ncases < 0) return fail(WLSQM_E_VALUE, "ncases must be >= 0");
    if (ncases > 0 && (!nk || !order || !knowns || !wm)) return fail(WLSQM_E_VALUE, "NULL metadata array");
    if (wlsqm_device_count() < 1) return fail(WLSQM_E_CUDA, "no CUDA device available (there is no CPU fallback)");
    if (device < 0 || device >= wlsqm_device_count()) return fail(WLSQM_E_VALUE, "bad device ordinal %d", device);

    wlsqm_solver* s = new (std::nothrow) wlsqm_solver();
    if (!s) return fail(WLSQM_E_MEMORY, "out of host memory");
    s->dim = dimension; s->device = device; s->algorithm = algorithm; s->do_sens = do_sens ? 1 : 0;
    s->max_iter = max_iter; s->debug = debug ? 1 : 0; s->ncases = ncases;
    // Uniform batches (every case with the same nk / order / knowns / weighting -- the usual ExpertSolver and
    // fit_*_many call) are recognised by one pass of comparisons and keep no per-case records at all.
    const bool all_same = scan_meta(ncases, nk, order, knowns, wm).uniform();
    const long long nrec = all_same ? std::min<long long>(ncases, 1) : ncases;
    try {
        s->hmeta.resize((size_t)nrec);
    } catch (...) {
        delete s;
        return fail(WLSQM_E_MEMORY, "out of host memory");
    }
    long long off = 0;
    for (long long i = 0; i < nrec; ++i) {
        const int no = number_of_dofs(dimension, order[i]);
        if (no < 0) { delete s; return fail(WLSQM_E_VALUE, "case %lld: order must be 0..4, got %d", i, order[i]); }
        if (nk[i] < 0) { delete s; return fail(WLSQM_E_VALUE, "case %lld: nk must be >= 0, got %d", i, nk[i]); }
        if (wm[i] != WLSQM_WEIGHT_UNIFORM && wm[i] != WLSQM_WEIGHT_CENTER) {
            delete s;
            return fail(WLSQM_E_VALUE, "case %lld: unknown weighting method %d", i, wm[i]);
        }
        CaseMeta& m = s->hmeta[(size_t)i];
        memset(&m, 0, sizeof m);
        m.knowns = knowns[i] & ((1LL << no) - 1);
        m.nkn = (signed char)__builtin_popcountll((unsigned long long)m.knowns);
        m.nk = nk[i]; m.no = (short)no; m.nr = (short)(no - m.nkn);
        m.order = (signed char)order[i]; m.wm = (signed char)wm[i];
        m.op_off = off;
        off += even((m.nk + m.nkn) * (int)m.nr);
        s->maxnk = std::max(s->maxnk, m.nk);
        s->maxno = std::max(s->maxno, no);
        s->maxnr = std::max(s->maxnr, (int)m.nr);
        s->maxnq = std::max(s->maxnq, m.nk + m.nkn);
        s->maxorder = std::max(s->maxorder, (int)m.order);
        s->maxnkn = std::max(s->maxnkn, (int)m.nkn);
        if (m.knowns) s->any_knowns = true;
        if (i > 0) {
            const CaseMeta& f = s->hmeta[0];
            if (m.nk != f.nk || m.order != f.order || m.knowns != f.knowns || m.wm != f.wm) s->uniform = false;
            if (m.no != f.no) s->uniform_no = false;
            if (m.nk != f.nk || m.order != f.order || m.nkn != f.nkn || m.wm != f.wm) s->geom_uniform = false;
        }
    }
    if (ncases > 0) s->last_nk_odd = (nk[ncases - 1] & 1) != 0;
    if (all_same) off *= ncases;
    s->op_total = off;
    if (ncases > 0) {
        s->uni = s->hmeta[0];
        s->uni.op_off = 0;
        s->op_stride = even((s->uni.nk + s->uni.nkn) * (int)s->uni.nr);
    }

    int rc = use_device(s);
    if (rc) { delete s; return rc; }
    {
        int smc = 0;   // (cudaGetDeviceProperties costs milliseconds; the one attribute is all that is needed)
        if (cudaDeviceGetAttribute(&smc, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && smc > 0) s->sm_count = smc;
        else cudaGetLastError();
    }
    cudaError_t e = cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { delete s; return fail(WLSQM_E_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e)); }
    s->own_stream = true;

    auto alloc = [&](void** p, size_t bytes) -> int {
        *p = nullptr;
        if (bytes == 0) return WLSQM_OK;
        cudaError_t e2 = dev_alloc(p, bytes);
        if (e2 != cudaSuccess) {
            cudaGetLastError();
            return fail(WLSQM_E_MEMORY, "device allocation of %zu bytes failed: %s", bytes, cudaGetErrorString(e2));
        }
        s->bytes_state += (long long)bytes;
        return WLSQM_OK;
    };
    rc = WLSQM_OK;
    if (!rc && !s->uniform) rc = alloc((void**)&s->dmeta, sizeof(CaseMeta) * (size_t)ncases);
    if (!rc && !s->uniform_no) rc = alloc((void**)&s->dorder, (size_t)ncases);
    if (!rc) rc = alloc((void**)&s->op, (size_t)s->op_total * 8);
    if (!rc) rc = alloc((void**)&s->fi_case, (size_t)ncases * s->maxno * 8);
    if (!rc) rc = alloc((void**)&s->xi_dev, (size_t)ncases * dimension * 8);
    if (!rc && s->debug) {
        s->as_stride = s->maxnr * s->maxnr;
        rc = alloc((void**)&s->As, (size_t)ncases * s->as_stride * 8);
    }
    if (!rc && algorithm == WLSQM_ALGO_ITERATIVE) rc = alloc((void**)&s->iters_dev, ((size_t)ncases + 1) * 4);
    std::vector<int> perm;
    if (!rc && !s->uniform_no && ncases >= env_int("WLSQM_PREP_BUCKET_MIN", 8192) && ncases < (1LL << 31)) {
        long long cnt[5] = {0, 0, 0, 0, 0};
        for (long long i = 0; i < ncases; ++i) ++cnt[s->hmeta[(size_t)i].order];
        for (int o = 0; o < 5; ++o) s->order_lo[o + 1] = s->order_lo[o] + cnt[o];
        long long at[5];
        for (int o = 0; o < 5; ++o) at[o] = s->order_lo[o];
        perm.resize((size_t)ncases);
        for (long long i = 0; i < ncases; ++i) perm[(size_t)at[s->hmeta[(size_t)i].order]++] = (int)i;
        rc = alloc((void**)&s->order_perm, (size_t)ncases * 4);
    }
    if (rc) { wlsqm_solver_destroy(s); return rc; }
    if (s->order_perm) cudaMemcpyAsync(s->order_perm, perm.data(), (size_t)ncases * 4, cudaMemcpyHostToDevice, s->stream);
    if (s->dmeta)
        cudaMemcpyAsync(s->dmeta, s->hmeta.data(), sizeof(CaseMeta) * (size_t)ncases, cudaMemcpyHostToDevice, s->stream);
    if (s->dorder) {
        std::vector<signed char> ho((size_t)ncases);
        for (long long i = 0; i < ncases; ++i) ho[(size_t)i] = s->hmeta[(size_t)i].order;
        cudaMemcpyAsync(s->dorder, ho.data(), (size_t)ncases, cudaMemcpyHostToDevice, s->stream);
        cudaStreamSynchronize(s->stream);
    }
    if (s->fi_case) cudaMemsetAsync(s->fi_case, 0, (size_t)ncases * s->maxno * 8, s->stream);
    e = cudaStreamSynchronize(s->stream);
    if (e != cudaSuccess) {
        wlsqm_solver_destroy(s);
        return fail(WLSQM_E_CUDA, "solver initialisation: %s", cudaGetErrorString(e));
    }
    *out = s;
    return WLSQM_OK;
}

int wlsqm_solver_destroy(wlsqm_solver_t* s) {
    if (!s) return WLSQM_OK;
    cudaSetDevice(s->device);
    // every stream that may still touch the solver's buffers, then the blocks go back to the pool unsynchronised
    if (s->stream) cudaStreamSynchronize(s->stream);
    if (s->s_in) cudaStreamSynchronize(s->s_in);
    if (s->s_out) cudaStreamSynchronize(s->s_out);
    if (!s->lender) {
        dev_free(s->dmeta); dev_free(s->dorder); dev_free(s->op); dev_free(s->xi_dev); dev_free(s->As); dev_free(s->order_perm);
        s->xk_keep.release();
    } else {
        s->xk_keep.p = nullptr; s->xk_keep.cap = 0;
    }
    dev_free(s->fi_case); dev_free(s->iters_dev); s->st_xk.release(); s->st_fk.release(); s->st_fi.release(); s->st_sens.release();
    s->st_x.release(); s->st_I.release(); s->st_out.release();
    s->hoods_dev.release(); s->hood_x.release(); s->hood_f.release(); s->hood_fk.release(); s->opx_coef.release();
    s->opx_runs.release(); s->opx_tmp.release();
    dev_free(s->hood_err);
    if (s->models_grid) { wlsqm_grid_destroy(s->models_grid); s->models_grid = nullptr; }
    if (s->own_stream && s->stream) cudaStreamDestroy(s->stream);
    if (s->s_in) cudaStreamDestroy(s->s_in);
    if (s->s_out) cudaStreamDestroy(s->s_out);
    for (cudaEvent_t e : s->events) cudaEventDestroy(e);
    cudaGetLastError();
    delete s;
    return WLSQM_OK;
}

// ExpertSolver(..., host=other) (expert.pyx:163-189, 243-263; infra.pyx:528-544): the guest borrows the host's
// geometry-dependent state -- here the operator blocks, per-case records, origins (and the kept xk of an iterative
// host) -- and owns only its solution copy, iteration counters and staging.  Several fields on one geometry then
// cost one set of operators.  The host must outlive the guest (the Python class keeps a reference).
int wlsqm_solver_create_guest(wlsqm_solver_t* host, int algorithm, int do_sens, int max_iter, wlsqm_solver_t** out) {
    if (!out) return fail(WLSQM_E_VALUE, "out is NULL");
    *out = nullptr;
    if (!host) return fail(WLSQM_E_VALUE, "NULL host solver");
    if (algorithm != WLSQM_ALGO_BASIC && algorithm != WLSQM_ALGO_ITERATIVE)
        return fail(WLSQM_E_VALUE, "Unknown algorithm specifier %d; see wlsqm.fitter.defs for valid specifiers ALGO_*", algorithm);
    if (algorithm == WLSQM_ALGO_ITERATIVE && host->algorithm != WLSQM_ALGO_ITERATIVE)
        return fail(WLSQM_E_VALUE, "an ALGO_ITERATIVE guest needs an ALGO_ITERATIVE host (the host keeps the geometry xk)");
    const wlsqm_solver* root = host->lender ? host->lender : host;
    wlsqm_solver* s = new (std::nothrow) wlsqm_solver();
    if (!s) return fail(WLSQM_E_MEMORY, "out of host memory");
    s->dim = root->dim; s->device = root->device; s->algorithm = algorithm; s->do_sens = do_sens ? 1 : 0;
    s->max_iter = max_iter; s->debug = root->debug; s->ncases = root->ncases;
    s->maxnk = root->maxnk; s->maxno = root->maxno; s->maxnr = root->maxnr; s->maxnq = root->maxnq;
    s->maxorder = root->maxorder; s->maxnkn = root->maxnkn;
    s->uniform = root->uniform; s->any_knowns = root->any_knowns; s->uniform_no = root->uniform_no; s->last_nk_odd = root->last_nk_odd;
    s->geom_uniform = root->geom_uniform;
    s->uni = root->uni; s->op_stride = root->op_stride; s->op_total = root->op_total;
    try {
        s->hmeta = root->hmeta;
    } catch (...) {
        delete s;
        return fail(WLSQM_E_MEMORY, "out of host memory");
    }
    s->sm_count = root->sm_count;
    s->lender = const_cast<wlsqm_solver*>(root);
    s->dmeta = root->dmeta; s->dorder = root->dorder; s->op = root->op; s->xi_dev = root->xi_dev;
    s->As = root->As; s->as_stride = root->as_stride;
    s->xk_keep.p = root->xk_keep.p; s->xk_keep.cap = 0;
    int rc = use_device(s);
    if (rc) { s->lender = nullptr; s->dmeta = nullptr; s->dorder = nullptr; s->op = nullptr; s->xi_dev = nullptr; s->As = nullptr; s->xk_keep.p = nullptr; delete s; return rc; }
    cudaError_t e = cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { wlsqm_solver_destroy(s); return fail(WLSQM_E_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e)); }
    s->own_stream = true;
    const size_t fb = (size_t)s->ncases * s->maxno * 8;
    if (fb && dev_alloc((void**)&s->fi_case, fb) != cudaSuccess) { cudaGetLastError(); wlsqm_solver_destroy(s); return fail(WLSQM_E_MEMORY, "cudaMalloc(%zu bytes) failed", fb); }
    s->bytes_state += (long long)fb;
    if (algorithm == WLSQM_ALGO_ITERATIVE) {
        const size_t ib = ((size_t)s->ncases + 1) * 4;
        if (dev_alloc((void**)&s->iters_dev, ib) != cudaSuccess) { cudaGetLastError(); wlsqm_solver_destroy(s); return fail(WLSQM_E_MEMORY, "cudaMalloc(%zu bytes) failed", ib); }
        s->bytes_state += (long long)ib;
    }
    if (s->fi_case) cudaMemsetAsync(s->fi_case, 0, fb, s->stream);
    e = cudaStreamSynchronize(s->stream);
    if (e != cudaSuccess) { wlsqm_solver_destroy(s); return fail(WLSQM_E_CUDA, "guest initialisation: %s", cudaGetErrorString(e)); }
    s->ready = root->ready;
    *out = s;
    return WLSQM_OK;
}

// guest.prepare(): nothing to compute -- the operators are the host's; the guest is ready when its host is
int wlsqm_solver_prepare_guest(wlsqm_solver_t* s) {
    if (!s || !s->lender) return fail(WLSQM_E_VALUE, "not a guest solver");
    if (!s->lender->ready) return fail(WLSQM_E_NOTREADY, "In guest mode, host must be in the ready state");
    int rc = use_device(s);
    if (rc) return rc;
    // the host may have re-prepared (and re-allocated its kept geometry) since the guest was created
    s->xk_keep.p = s->lender->xk_keep.p;
    if (s->models_grid) { wlsqm_grid_destroy(s->models_grid); s->models_grid = nullptr; }
    CU(cudaStreamSynchronize(s->lender->stream));     // the host's prepare may still be in flight on its stream
    s->ready = true;
    return WLSQM_OK;
}

int wlsqm_solver_set_stream(wlsqm_solver_t* s, void* cuda_stream) {
    if (!s) return fail(WLSQM_E_VALUE, "NULL solver");
    cudaStream_t next = (cudaStream_t)cuda_stream;
    if (!s->own_stream && s->stream == next) return WLSQM_OK;
    cudaSetDevice(s->device);
    if (s->own_stream && s->stream) {
        cudaStreamSynchronize(s->stream);
        cudaStreamDestroy(s->stream);
    } else {
        // work queued on the previous caller stream (a prepare, say) must be visible to what follows on the new one
        CU(order_streams(s->stream, next));
    }
    s->stream = next;
    s->own_stream = false;
    return WLSQM_OK;
}

// ---- fused result gather over peer memory (multi-GPU; SURVEY.md 8e) -----------------------------------------------
// One process per GPU.  Every rank allocates its copy of the GLOBAL solution array with wlsqm_peer_alloc and publishes
// the 64-byte IPC handle; the others open it (wlsqm_peer_open).  wlsqm_solver_set_gather hands the solver the base
// pointers of all copies: from then on solve() stores every row it computes into each of them (its own included),
// i.e. the all-gather of fi happens inside the solve kernel, tile by tile, over NVLink.  The ranks still need one
// synchronisation per step before they read rows written by their peers (any stream-ordered barrier).
int wlsqm_peer_alloc(int device, int64_t bytes, void** ptr, void* ipc_handle_64) {
    if (!ptr || !ipc_handle_64 || bytes <= 0) return fail(WLSQM_E_VALUE, "wlsqm_peer_alloc: bad argument");
    *ptr = nullptr;
    if (wlsqm_device_count() < 1) return fail(WLSQM_E_CUDA, "no CUDA device available (there is no CPU fallback)");
    CU(cudaSetDevice(device));
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, (size_t)bytes);      // (IPC needs a plain allocation, not a block of the stream-ordered pool)
    if (e != cudaSuccess) { cudaGetLastError(); return fail(WLSQM_E_MEMORY, "cudaMalloc(%lld bytes) failed: %s", (long long)bytes, cudaGetErrorString(e)); }
    cudaIpcMemHandle_t h;
    e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaGetLastError(); cudaFree(p); return fail(WLSQM_E_CUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e)); }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    memcpy(ipc_handle_64, &h, 64);
    CU(cudaMemset(p, 0, (size_t)bytes));
    *ptr = p;
    return WLSQM_OK;
}
int wlsqm_peer_open(int device, const void* ipc_handle_64, void** ptr) {
    if (!ptr || !ipc_handle_64) return fail(WLSQM_E_VALUE, "wlsqm_peer_open: bad argument");
    *ptr = nullptr;
    CU(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    memcpy(&h, ipc_handle_64, 64);
    cudaError_t e = cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) { cudaGetLastError(); *ptr = nullptr; return fail(WLSQM_E_CUDA, "cudaIpcOpenMemHandle: %s", cudaGetErrorString(e)); }
    return WLSQM_OK;
}
int wlsqm_peer_close(void* ptr) {
    if (ptr && cudaIpcCloseMemHandle(ptr) != cudaSuccess) cudaGetLastError();
    return WLSQM_OK;
}
int wlsqm_peer_free(void* ptr) {
    if (ptr && cudaFree(ptr) != cudaSuccess) cudaGetLastError();
    return WLSQM_OK;
}
int wlsqm_solver_keep_solution(wlsqm_solver_t* s, int keep) {
    if (!s) return fail(WLSQM_E_VALUE, "NULL solver");
    s->keep_solution = keep != 0;
    return WLSQM_OK;
}

int wlsqm_solver_set_gather(wlsqm_solver_t* s, int ntargets, void* const* bases, int64_t row0, int64_t row_stride) {
    if (!s) return fail(WLSQM_E_VALUE, "NULL solver");
    if (ntargets < 0 || ntargets > WLSQM_MAX_PEERS) return fail(WLSQM_E_VALUE, "between 0 and %d gather targets", WLSQM_MAX_PEERS);
    if (ntargets > 0 && (!bases || row_stride < s->maxno || row0 < 0)) return fail(WLSQM_E_VALUE, "wlsqm_solver_set_gather: bad layout");
    for (int p = 0; p < ntargets; ++p)
        if (!bases[p]) return fail(WLSQM_E_VALUE, "wlsqm_solver_set_gather: NULL target");
    s->ngather = ntargets;
    for (int p = 0; p < WLSQM_MAX_PEERS; ++p) s->gather[p] = p < ntargets ? (double*)bases[p] : nullptr;
    s->gather_row0 = row0; s->gather_s0 = row_stride;
    return WLSQM_OK;
}

int wlsqm_set_caller_stream(void* cuda_stream) {
    set_caller_stream((cudaStream_t)cuda_stream);
    return WLSQM_OK;
}

int wlsqm_solver_synchronize(wlsqm_solver_t* s) {
    if (!s) return fail(WLSQM_E_VALUE, "NULL solver");
    int rc = use_device(s);
    if (rc) return rc;
    CU(cudaStreamSynchronize(s->stream));
    return WLSQM_OK;
}

int wlsqm_solver_prepare(wlsqm_solver_t* s, const double* xi, int64_t xi_s0, const double* xk, int64_t xk_s0,
                         int64_t xk_s1) {
    if (!s) return fail(WLSQM_E_VALUE, "NULL solver");
    if (s->lender) return wlsqm_solver_prepare_guest(s);
    s->ready = false;
    s->hoods_current = false;   // (prepare_hoods sets it again once its own prepare has succeeded)
    if (s->models_grid) { wlsqm_grid_destroy(s->models_grid); s->models_grid = nullptr; }   // the origins may move
    if (s->ncases == 0) { s->ready = true; return WLSQM_OK; }
    if (!xi || !xk) return fail(WLSQM_E_VALUE, "xi and xk must not be NULL");
    int rc = use_device(s);
    if (rc) return rc;
    const int dim = s->dim;
    const long long n = s->ncases;
    const bool iter = s->algorithm == WLSQM_ALGO_ITERATIVE;

    // origins: always kept (interpolate and ALGO_ITERATIVE need them)
    rc = to_dense(s->xi_dev, xi, n, dim, xi_s0, s->stream);
    if (rc) return rc;

    const double* xk_use = xk;
    long long s0 = xk_s0, s1 = xk_s1;
    const bool xk_dev = is_device_ptr(xk);
    if (!xk_dev || iter) {
        DevBuf& buf = iter ? s->xk_keep : s->st_xk;
        const long long row = (long long)s->maxnk * dim;
        rc = buf.reserve((size_t)n * row * 8);
        if (rc) return rc;
        if (xk_s1 == dim) {
            rc = stage_in(s->device, (double*)buf.p, xk, n, row, xk_s0, s->stream);
            if (rc) return rc;
        } else if (xk_dev) {
            gather3_kernel<<<s->sm_count * 8, 256, 0, s->stream>>>((double*)buf.p, xk, n, s->maxnk, dim, xk_s0, xk_s1, 1);
            CU(cudaGetLastError());
        } else {
            return fail(WLSQM_E_VALUE, "host xk must have contiguous neighbour rows (stride %lld != %d)", (long long)xk_s1, dim);
        }
        xk_use = (const double*)buf.p;
        s0 = row;
        s1 = dim;
    }

    LaunchCfg L;
    PrepRegParams R{};
    R.meta = s->dmeta; R.uni = s->uni; R.op_stride = s->op_stride; R.ncases = n;
    R.geom_uniform = s->geom_uniform ? 1 : 0;
    R.xi = s->xi_dev; R.xi_s0 = dim;
    R.xk = xk_use; R.xk_s0 = s0; R.xk_s1 = s1;
    R.op = s->op; R.As = s->As; R.as_stride = s->as_stride;
    const char* ksel = getenv("WLSQM_PREP_KERNEL");
    const bool want_smem = ksel && !strcmp(ksel, "smem");
    if (!want_smem && config_prepare_reg(s, R, L)) {
        if (s->order_perm && env_int("WLSQM_PREP_BUCKETS", 1) != 0) {
            // mixed orders: one launch per order over its case list, each with the kernel instantiated for that order
            // (an order-2 fit in the order-4 kernel pays for 16-wide rows; measured in profiles/README.md)
            for (int o = 0; o < 5; ++o) {
                const long long cnt = s->order_lo[o + 1] - s->order_lo[o];
                if (cnt < 1) continue;
                PrepRegParams Ro = R;
                LaunchCfg Lo;
                Ro.perm = s->order_perm + s->order_lo[o];
                Ro.ncases = cnt;
                if (!config_prepare_reg(s, Ro, Lo, false, o, cnt)) return fail(WLSQM_E_VALUE, "prepare: no launch shape for order %d", o);
                CU(launch_prepare_reg(dim, o, Ro, Lo.blocks, Lo.threads, Lo.smem, s->stream));
            }
        } else {
            CU(launch_prepare_reg(dim, s->maxorder, R, L.blocks, L.threads, L.smem, s->stream));
        }
    } else {
        PrepareParams P{};
        P.meta = s->dmeta; P.uni = s->uni; P.op_stride = s->op_stride; P.ncases = n;
        P.xi = s->xi_dev; P.xi_s0 = dim;
        P.xk = xk_use; P.xk_s0 = s0; P.xk_s1 = s1;
        P.op = s->op; P.As = s->As; P.as_stride = s->as_stride;
        rc = config_prepare(s, P, L);
        if (rc) return rc;
        CU(launch_prepare_smem(dim, P, L.blocks, L.threads, L.smem, s->stream));
    }
    if (!xk_dev) {
        // the call owns the host array only until it returns
        CU(cudaStreamSynchronize(s->stream));
        if (!iter) s->st_xk.release();
    }
    s->ready = true;
    return WLSQM_OK;
}

int wlsqm_solver_solve(wlsqm_solver_t* s, const double* fk, int64_t fk_s0, int64_t fk_s1, double* fi, int64_t fi_s0,
                       double* sens, int64_t sens_s0, int64_t sens_s1, int32_t* iters_out) {
    if (!s) return fail(WLSQM_E_VALUE, "NULL solver");
    if (!s->ready) return fail(WLSQM_E_NOTREADY, "Solver is not in the ready state; prepare() must be called before solve()");
    if (iters_out) *iters_out = 0;
    if (s->ncases == 0) return WLSQM_OK;
    if (!fk || !fi) return fail(WLSQM_E_VALUE, "fk and fi must not be NULL");
    if (s->do_sens && !sens) return fail(WLSQM_E_VALUE, "sens must be given when do_sens is set");
    int rc = use_device(s);
    if (rc) return rc;
    const long long n = s->ncases;
    const bool iter = s->algorithm == WLSQM_ALGO_ITERATIVE;
    const bool fk_dev = is_device_ptr(fk), fi_dev = is_device_ptr(fi);
    const bool sens_dev = s->do_sens ? (is_device_ptr(sens) != 0) : true;
    cudaStream_t st = s->stream;

    SolveParams P{};
    solve_params(s, P);
    if (iter) CU(cudaMemsetAsync(s->iters_dev, 0, 4, st));
    P.fi_case = s->fi_case; P.fi_case_ld = s->maxno;
    P.ngather = s->ngather;
    for (int p = 0; p < s->ngather; ++p) P.gather[p] = s->gather[p];
    P.gather_row0 = s->gather_row0; P.gather_s0 = s->gather_s0;
    P.gather_full = (s->ngather > 0 && s->gather_s0 % 16 == 0 && s->gather_s0 <= 32 && s->gather_s0 > s->maxno) ? 1 : 0;

    // ---- device-side views of the arguments (host arrays get dense device mirrors) -------------------
    const bool staged = !fk_dev || !fi_dev || !sens_dev;
    if (fk_dev) {
        P.fk = fk; P.fk_s0 = fk_s0; P.fk_s1 = fk_s1;
    } else {
        if (fk_s1 != 1 && s->maxnk > 1) return fail(WLSQM_E_VALUE, "host fk must have unit stride on its last axis");
        rc = s->st_fk.reserve((size_t)n * s->maxnk * 8);
        if (rc) return rc;
        P.fk = (const double*)s->st_fk.p; P.fk_s0 = s->maxnk; P.fk_s1 = 1;
    }
    bool deferred = false;
    s->fi_case_valid = true;
    if (fi_dev) {
        P.fi_in = fi; P.fi_in_s0 = fi_s0;
        // the caller's fk may be a view into fi (expert.pyx:548-555): then write back only after all cases are solved
        bool alias = false;
        if (fk_dev) {
            if (fk_s0 < 0 || fk_s1 < 0 || fi_s0 < 0) alias = true;
            else
                alias = ranges_overlap(fk, ((n - 1) * fk_s0 + (long long)(s->maxnk - 1) * fk_s1 + 1) * 8, fi,
                                       ((n - 1) * fi_s0 + s->maxno) * 8);
        }
        if (alias) deferred = true;
        else { P.fi_out = fi; P.fi_out_s0 = fi_s0; }
        if (!s->keep_solution && !deferred) P.fi_case = nullptr;
        s->fi_case_valid = P.fi_case != nullptr;
    } else if (s->any_knowns) {
        rc = s->st_fi.reserve((size_t)n * s->maxno * 8);
        if (rc) return rc;
        P.fi_in = (const double*)s->st_fi.p; P.fi_in_s0 = s->maxno;
    }
    const long long plane = (long long)s->maxnk * s->maxno;
    // host sens: the kernel writes each chunk of cases into one of two rotating device buffers (2 x chunk x nk x no
    // doubles -- not a mirror of the whole array, which is 67 GB for BASELINE.json configs[2]); a chunk goes back to the
    // host while the next one is being computed
    const bool sens_host = s->do_sens && !sens_dev;
    if (s->do_sens && sens_dev) { P.sens = sens; P.sens_s0 = sens_s0; P.sens_s1 = sens_s1; }
    // page-locked, dense, uniform: straight asynchronous copies; anything else (ordinary numpy memory, pitched rows,
    // per-case nk / no) goes through the page-locked ring and is scattered by the host threads
    const bool sens_direct = sens_host && s->uniform && s->uni.nk == s->maxnk && sens_s1 == s->maxno && sens_s0 == plane &&
                             !is_pageable_host(sens);
    const bool sens_drain = sens_host && !sens_direct;
    constexpr int SENS_BUFS = 2;

    // ---- chunked pipeline: H2D of chunk i+1, kernel of chunk i and D2H of chunk i-1 overlap ------------
    // (device-resident arguments: one chunk, everything on the solver's stream, no synchronisation)
    long long chunk = n;
    cudaStream_t s_in = st, s_out = st;
    if (staged) {
        chunk = std::max<long long>(1024, env_int("WLSQM_SOLVE_CHUNK", 65536));
        if (sens_host) {
            // a chunk of sens must fit a share of the ring slot granularity and keep the buffers modest
            const long long cap = std::max<long long>(256, (long long)((1ull << 30) / ((size_t)std::max<long long>(plane, 1) * 8)));
            chunk = std::min(chunk, cap);
            rc = s->st_sens.reserve((size_t)SENS_BUFS * (size_t)std::min(chunk, n) * plane * 8);
            if (rc) return rc;
        }
        if (!s->s_in) CU(cudaStreamCreateWithFlags(&s->s_in, cudaStreamNonBlocking));
        if (!s->s_out) CU(cudaStreamCreateWithFlags(&s->s_out, cudaStreamNonBlocking));
        s_in = s->s_in; s_out = s->s_out;
        const size_t nev = 2 * (size_t)((n + chunk - 1) / chunk) + 1 + SENS_BUFS;
        while (s->events.size() < nev) {
            cudaEvent_t e;
            CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            s->events.push_back(e);
        }
        // the copy streams must not run ahead of work already queued on the solver's stream
        CU(cudaEventRecord(s->events[nev - 1], st));
        CU(cudaStreamWaitEvent(s_in, s->events[nev - 1], 0));
    }
    // ordinary (pageable) numpy arrays: host threads copy through rings of page-locked slots (wlsqm_host.h)
    const bool fk_bounce = !fk_dev && n * s->maxnk * 8 >= BOUNCE_MIN_BYTES && is_pageable_host(fk) &&
                           (size_t)s->maxnk * 8 <= BOUNCE_SLOT_BYTES && env_int("WLSQM_BOUNCE", 1) != 0;
    const bool fi_bounce = !fi_dev && s->uniform_no && (fk_bounce || n * s->maxno * 8 >= BOUNCE_MIN_BYTES) &&
                           is_pageable_host(fi) && env_int("WLSQM_BOUNCE", 1) != 0 &&
                           (size_t)chunk * s->uni.no * 8 <= BOUNCE_SLOT_BYTES;
    struct RingGuard {
        bool on = false;
        ~RingGuard() { if (on) bounce_unlock(); }
    } ring_guard;
    const bool fi_scatter = !fi_dev && !s->uniform_no;       // per-case row lengths: unpacked by the host threads
    BouncePair* rings = nullptr;
    if (fk_bounce || fi_bounce || sens_drain || fi_scatter) {
        bounce_lock();
        ring_guard.on = true;
        rings = &bounce_rings(s->device);
    }
    struct PendingOut { int slot; long long c0, rows; };
    std::vector<PendingOut> pend;
    auto finish_oldest = [&]() -> int {
        const PendingOut p = pend.front();
        pend.erase(pend.begin());
        CU(d2h_bounced_finish(rings->out, p.slot, fi + p.c0 * fi_s0, fi_s0, p.rows, s->uni.no));
        return WLSQM_OK;
    };
    // one chunk of sens from its device buffer to the caller's host array (first nk_j rows x no_j columns of every case)
    struct SensChunk { long long c0 = 0, rows = 0; const double* buf = nullptr; bool live = false; } sens_prev;
    auto drain_sens = [&](const SensChunk& ch) -> int {
        while (!pend.empty()) { int r2 = finish_oldest(); if (r2) return r2; }      // (the ring is shared with the fi pieces)
        const cudaError_t e2 = d2h_pieces(rings->out, ch.buf, ch.rows, plane, s_out, [&](const double* piece, long long r0, long long nr) {
            par_for((size_t)nr, [&](size_t lo, size_t hi) {
                for (size_t r = lo; r < hi; ++r) {
                    const long long i = ch.c0 + r0 + (long long)r;
                    const CaseMeta& m = s->hmeta.size() > (size_t)i ? s->hmeta[(size_t)i] : s->uni;
                    if (m.nr < 1) continue;     // silent no-op case: sens untouched (impl.pyx:742)
                    const double* src = piece + r * plane;
                    double* dst = sens + i * sens_s0;
                    if (m.no == s->maxno && sens_s1 == s->maxno) memcpy(dst, src, (size_t)m.nk * m.no * 8);
                    else
                        for (int k = 0; k < m.nk; ++k) memcpy(dst + (long long)k * sens_s1, src + (size_t)k * s->maxno, (size_t)m.no * 8);
                }
            });
        });
        if (e2 != cudaSuccess) return fail(WLSQM_E_CUDA, "device -> host staging of sens: %s", cudaGetErrorString(e2));
        return WLSQM_OK;
    };
    LaunchCfg L;
    size_t ev = 0;
    long long chunk_index = 0;
    const size_t sens_ev0 = s->events.size() >= (size_t)SENS_BUFS ? s->events.size() - 1 - SENS_BUFS : 0;   // (staged: reserved above)
    for (long long c0 = 0; c0 < n; c0 += chunk, ++chunk_index) {
        const long long c1 = std::min(n, c0 + chunk), rows = c1 - c0;
        const int sb = (int)(chunk_index % SENS_BUFS);
        double* sens_buf = nullptr;
        if (sens_host) {
            sens_buf = (double*)s->st_sens.p + (size_t)sb * (size_t)std::min(chunk, n) * plane;
            // the kernel indexes sens by the global case number: bias the base so that case c0 lands at the buffer's start
            P.sens = reinterpret_cast<double*>(reinterpret_cast<uintptr_t>(sens_buf) - (uintptr_t)c0 * (uintptr_t)plane * 8u);
            P.sens_s0 = plane; P.sens_s1 = s->maxno;
            if (sens_direct && chunk_index >= SENS_BUFS) CU(cudaStreamWaitEvent(st, s->events[sens_ev0 + sb], 0));   // its last copy out is done
        }
        if (fk_bounce) {
            CU(h2d_bounced(rings->in, (double*)s->st_fk.p + c0 * s->maxnk, fk + c0 * fk_s0, rows, s->maxnk, fk_s0, s_in));
        } else if (!fk_dev) {
            rc = to_dense((double*)s->st_fk.p + c0 * s->maxnk, fk + c0 * fk_s0, rows, s->maxnk, fk_s0, s_in);
            if (rc) return rc;
        }
        if (!fi_dev && s->any_knowns) {
            rc = to_dense((double*)s->st_fi.p + c0 * s->maxno, fi + c0 * fi_s0, rows, s->maxno, fi_s0, s_in);
            if (rc) return rc;
        }
        if (staged) {
            CU(cudaEventRecord(s->events[ev], s_in));
            CU(cudaStreamWaitEvent(st, s->events[ev], 0));
            ++ev;
        }
        P.case_lo = c0;
        P.ncases = c1;
        if (pack_eligible(s)) {
            rc = launch_solve_split(P, false, [&](long long r) { return config_solve_pack(s, P, L, r); },
                                    [&] { return launch_solve_pack(P, L.blocks, L.threads, L.smem, st); });
        } else {
            rc = launch_solve_split(P, fk_dev && s->last_nk_odd && c1 == n, [&](long long r) { return config_solve(s, P, L, r); },
                                    [&] { return launch_solve(s->dim, P, L.blocks, L.threads, L.smem, st); });
        }
        if (rc) return rc;
        if (sens_drain) {
            // the previous chunk goes to the host while this one is being computed (its copies were queued on s_out
            // before s_out is told to wait for this chunk's kernel)
            if (sens_prev.live) { rc = drain_sens(sens_prev); if (rc) return rc; }
            sens_prev.c0 = c0; sens_prev.rows = rows; sens_prev.buf = sens_buf; sens_prev.live = true;
        }
        if (staged) {
            CU(cudaEventRecord(s->events[ev], st));
            CU(cudaStreamWaitEvent(s_out, s->events[ev], 0));
            ++ev;
        }
        if (fi_bounce) {
            if ((int)pend.size() >= BOUNCE_SLOTS - 1) { rc = finish_oldest(); if (rc) return rc; }
            const int slot = d2h_bounced_begin(rings->out, s->fi_case + c0 * s->maxno, s->maxno, rows, s->uni.no, s_out);
            if (slot < 0) return fail(WLSQM_E_CUDA, "device -> host staging: %s", cudaGetErrorString((cudaError_t)(-slot)));
            pend.push_back(PendingOut{slot, c0, rows});
        } else if (!fi_dev && s->uniform_no) {
            rc = from_dense(fi + c0 * fi_s0, fi_s0, s->fi_case + c0 * s->maxno, s->maxno, rows, s->uni.no, s_out);
            if (rc) return rc;
        }
        if (sens_direct) {
            CU(cudaMemcpyAsync(sens + c0 * plane, sens_buf, (size_t)rows * plane * 8, cudaMemcpyDeviceToHost, s_out));
            CU(cudaEventRecord(s->events[sens_ev0 + sb], s_out));
        }
    }
    if (sens_drain && sens_prev.live) { rc = drain_sens(sens_prev); if (rc) return rc; }
    while (!pend.empty()) { rc = finish_oldest(); if (rc) return rc; }
    if (deferred) CU(launch_scatter_fi(s->dmeta, s->uni, n, s->fi_case, s->maxno, fi, fi_s0, st));

    // ---- fi with per-case row lengths: pieces through the page-locked ring, scattered by the host threads ----------
    if (fi_scatter) {
        const int ld = s->maxno;
        const cudaError_t e2 = d2h_pieces(rings->out, s->fi_case, n, ld, s_out, [&](const double* piece, long long r0, long long nr) {
            par_for((size_t)nr, [&](size_t lo, size_t hi) {
                for (size_t r = lo; r < hi; ++r) {
                    const long long i = r0 + (long long)r;
                    memcpy(fi + i * fi_s0, piece + r * ld, (size_t)s->hmeta[(size_t)i].no * 8);
                }
            });
        });
        if (e2 != cudaSuccess) return fail(WLSQM_E_CUDA, "device -> host staging of fi: %s", cudaGetErrorString(e2));
    }
    int32_t it = 0;
    if (iter) CU(cudaMemcpyAsync(&it, s->iters_dev, 4, cudaMemcpyDeviceToHost, st));
    if (staged) CU(cudaStreamSynchronize(s_out));
    if (iter || staged) CU(cudaStreamSynchronize(st));
    if (iters_out) *iters_out = it;
    return WLSQM_OK;
}

int wlsqm_solver_iterations(wlsqm_solver_t* s, int32_t* out) {
    if (!s || !out) return fail(WLSQM_E_VALUE, "NULL argument");
    if (s->algorithm != WLSQM_ALGO_ITERATIVE) {
        memset(out, 0, (size_t)s->ncases * 4);
        return WLSQM_OK;
    }
    int rc = use_device(s);
    if (rc) return rc;
    CU(cudaMemcpyAsync(out, s->iters_dev + 1, (size_t)s->ncases * 4, cudaMemcpyDeviceToHost, s->stream));
    CU(cudaStreamSynchronize(s->stream));
    return WLSQM_OK;
}

int wlsqm_solver_interpolate(wlsqm_solver_t* s, const double* x, int64_t x_s0, const int64_t* I, int64_t nx, int diff,
                             double* out, int64_t out_s0) {
    if (!s) return fail(WLSQM_E_VALUE, "NULL solver");
    if (!s->ready) return fail(WLSQM_E_NOTREADY, "Solver is not in the ready state; prepare() must be called first");
    if (nx == 0) return WLSQM_OK;
    if (!x || !I || !out) return fail(WLSQM_E_VALUE, "x, I and out must not be NULL");
    if (!s->fi_case_valid) return fail(WLSQM_E_NOTREADY, "the solver keeps no copy of the solution (wlsqm_solver_keep_solution(s, 0)); solve() again with the copy enabled");
    const int size = number_of_dofs(s->dim, 4);
    if (diff != WLSQM_DIFF_ALL && (diff < 0 || diff >= size)) return fail(WLSQM_E_VALUE, "invalid diff %d", diff);
    int rc = use_device(s);
    if (rc) return rc;
    cudaStream_t st = s->stream;
    const bool x_dev = is_device_ptr(x), I_dev = is_device_ptr(I), out_dev = is_device_ptr(out);
    const long long ow = diff == WLSQM_DIFF_ALL ? s->maxno : 1;
    InterpParams P{};
    P.dim = s->dim; P.nx = nx; P.diff = diff; P.nmodels = s->ncases;
    P.xi = s->xi_dev; P.xi_s0 = s->dim; P.fi = s->fi_case; P.fi_s0 = s->maxno;
    P.order = s->dorder; P.order_uniform = s->uni.order;
    if (x_dev) { P.x = x; P.x_s0 = x_s0; }
    else {
        rc = s->st_x.reserve((size_t)nx * s->dim * 8);
        if (rc) return rc;
        rc = stage_in(s->device, (double*)s->st_x.p, x, nx, s->dim, x_s0, st);
        if (rc) return rc;
        P.x = (const double*)s->st_x.p; P.x_s0 = s->dim;
    }
    if (I_dev) P.I = (const long long*)I;
    else {
        rc = s->st_I.reserve((size_t)nx * 8);
        if (rc) return rc;
        rc = stage_in(s->device, (double*)s->st_I.p, reinterpret_cast<const double*>(I), nx, 1, 1, st);   // (8-byte items)
        if (rc) return rc;
        P.I = (const long long*)s->st_I.p;
    }
    if (out_dev) { P.out = out; P.out_s0 = diff == WLSQM_DIFF_ALL ? out_s0 : 1; }
    else {
        rc = s->st_out.reserve((size_t)nx * ow * 8);
        if (rc) return rc;
        if (diff == WLSQM_DIFF_ALL && !s->uniform_no) CU(cudaMemsetAsync(s->st_out.p, 0, (size_t)nx * ow * 8, st));
        P.out = (double*)s->st_out.p; P.out_s0 = ow;
    }
    P.stage_no = (diff == WLSQM_DIFF_ALL && s->uniform_no && P.out_s0 == s->uni.no) ? s->uni.no : 0;
    CU(launch_interpolate(P, st));
    if (!out_dev) {
        if (diff == WLSQM_DIFF_ALL) rc = stage_out(s->device, out, out_s0, (const double*)s->st_out.p, ow, nx, ow, st);
        else rc = stage_out(s->device, out, 1, (const double*)s->st_out.p, 1, nx, 1, st);
        if (rc) return rc;
    }
    if (!x_dev || !I_dev || !out_dev) CU(cudaStreamSynchronize(st));
    return WLSQM_OK;
}

int wlsqm_solver_conds(wlsqm_solver_t* s, double* out) {
    if (!s || !out) return fail(WLSQM_E_VALUE, "NULL argument");
    if (!s->ready) return fail(WLSQM_E_NOTREADY, "Solver is not in the ready state; prepare() must be called before conds()");
    if (!s->debug) return fail(WLSQM_E_NOTREADY, "Not in debug mode; condition number data has not been computed");
    if (s->ncases == 0) return WLSQM_OK;
    int rc = use_device(s);
    if (rc) return rc;
    const bool out_dev = is_device_ptr(out);
    double* d = out;
    if (!out_dev) {
        rc = s->st_out.reserve((size_t)s->ncases * 8);
        if (rc) return rc;
        d = (double*)s->st_out.p;
    }
    CU(launch_cond(s->maxnr, s->ncases, s->dmeta, s->uni, s->As, s->as_stride, d, s->stream));
    if (!out_dev) CU(cudaMemcpyAsync(out, d, (size_t)s->ncases * 8, cudaMemcpyDeviceToHost, s->stream));
    CU(cudaStreamSynchronize(s->stream));
    return WLSQM_OK;
}

int wlsqm_solver_memory(wlsqm_solver_t* s, int64_t* used, int64_t* total) {
    if (!s) return fail(WLSQM_E_VALUE, "NULL solver");
    if (used) *used = s->bytes_state;
    if (total) *total = s->bytes_state + staging_bytes(s);
    return WLSQM_OK;
}

int wlsqm_solver_get_fi(wlsqm_solver_t* s, double* out, int64_t out_s0) {
    if (!s || !out) return fail(WLSQM_E_VALUE, "NULL argument");
    if (s->ncases == 0) return WLSQM_OK;
    if (!s->fi_case_valid) return fail(WLSQM_E_NOTREADY, "the solver keeps no copy of the solution (wlsqm_solver_keep_solution(s, 0)); solve() again with the copy enabled");
    int rc = use_device(s);
    if (rc) return rc;
    rc = from_dense(out, out_s0, s->fi_case, s->maxno, s->ncases, s->maxno, s->stream);
    if (rc) return rc;
    CU(cudaStreamSynchronize(s->stream));
    return WLSQM_OK;
}

int wlsqm_gather_hoods(const double* src, int64_t src_s0, int w, int64_t nsrc, const int32_t* idx, int64_t idx_s0, int64_t n,
                       int k, double* dst, int device, void* cuda_stream) {
    if (n == 0 || k == 0 || w == 0) return WLSQM_OK;
    if (!src || !idx || !dst) return fail(WLSQM_E_VALUE, "NULL argument");
    if (!is_device_ptr(src) || !is_device_ptr(idx) || !is_device_ptr(dst))
        return fail(WLSQM_E_VALUE, "wlsqm_gather_hoods works on device arrays");
    CU(cudaSetDevice(device));
    const long long total = (long long)n * k * w;
    const unsigned blocks = (unsigned)std::min<long long>((total + 255) / 256, 148LL * 32);
    // asynchronous on the caller's stream: an index outside [0, nsrc) yields NaN (no flag can be reported without a sync)
    gather_hoods_kernel<<<blocks, 256, 0, (cudaStream_t)cuda_stream>>>(src, src_s0, w, idx, idx_s0, n, k, dst, nsrc, nullptr,
                                                                      -1, nullptr);
    CU(cudaGetLastError());
    return WLSQM_OK;
}

// ExpertSolver.prepare with the neighbourhoods given as index lists into a point array: xk = x[hoods] is
// gathered on the device (the caller-side gather of examples/expertsolver_example.py:59-66).
int wlsqm_solver_prepare_hoods(wlsqm_solver_t* s, const double* x, int64_t x_s0, int64_t npoints, const int32_t* hoods,
                               int64_t hoods_s0, const double* xi, int64_t xi_s0) {
    if (!s) return fail(WLSQM_E_VALUE, "NULL solver");
    s->hoods_current = false;   // until the new neighbour lists and the operators built from them are both in place
    if (s->ncases == 0) {
        const int rc0 = wlsqm_solver_prepare(s, x, x_s0, x, 0, 0);
        if (rc0) return rc0;
        s->hood_points = npoints;
        s->hoods_current = true;
        return WLSQM_OK;
    }
    if (!x || !hoods) return fail(WLSQM_E_VALUE, "x and hoods must not be NULL");
    if (!xi && npoints < s->ncases) return fail(WLSQM_E_VALUE, "without xi, x must hold one point per case");
    int rc = use_device(s);
    if (rc) return rc;
    const int dim = s->dim;
    const long long n = s->ncases;
    cudaStream_t st = s->stream;
    const double* xd = x;
    long long xs0 = x_s0;
    if (!is_device_ptr(x)) {
        rc = s->hood_x.reserve((size_t)npoints * dim * 8);
        if (rc) return rc;
        rc = to_dense((double*)s->hood_x.p, x, npoints, dim, x_s0, st);
        if (rc) return rc;
        xd = (const double*)s->hood_x.p;
        xs0 = dim;
    }
    rc = s->hoods_dev.reserve((size_t)n * s->maxnk * 4);
    if (rc) return rc;
    CU(cudaMemcpy2DAsync(s->hoods_dev.p, (size_t)s->maxnk * 4, hoods, (size_t)hoods_s0 * 4, (size_t)s->maxnk * 4, (size_t)n,
                         cudaMemcpyDefault, st));
    s->hood_points = npoints;
    rc = s->st_xk.reserve((size_t)n * s->maxnk * dim * 8);
    if (rc) return rc;
    if (!s->hood_err) {
        if (dev_alloc((void**)&s->hood_err, 4) != cudaSuccess) { cudaGetLastError(); return fail(WLSQM_E_MEMORY, "device allocation failed"); }
    }
    CU(cudaMemsetAsync(s->hood_err, 0, 4, st));
    CU(gather_hoods(s, xd, xs0, dim, s->maxnk, (double*)s->st_xk.p, s->hood_err));
    const double* xi_use = xi ? xi : xd;
    const long long xi_use_s0 = xi ? xi_s0 : xs0;
    rc = wlsqm_solver_prepare(s, xi_use, xi_use_s0, (const double*)s->st_xk.p, (long long)s->maxnk * dim, dim);
    if (rc) return rc;
    int herr = 0;
    CU(cudaMemcpyAsync(&herr, s->hood_err, 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (herr) {
        // the reference's caller-side gather x[hoods] raises IndexError here (examples/expertsolver_example.py:66)
        s->ready = false;
        s->hoods_dev.release();
        return fail(WLSQM_E_VALUE, "hoods: a neighbour index among the first nk[i] of some case lies outside [0, %lld)", (long long)npoints);
    }
    s->st_xk.release();      // (ALGO_ITERATIVE keeps its own copy of the geometry)
    s->hood_x.release();
    s->hoods_current = true;
    return WLSQM_OK;
}

// ExpertSolver.solve with the data given per point: fk = f[hoods] is gathered on the device, so that a time step
// moves one value per point to the GPU instead of one per (point, neighbour).
int wlsqm_solver_solve_hoods(wlsqm_solver_t* s, const double* f, int64_t f_s0, double* fi, int64_t fi_s0, double* sens,
                             int64_t sens_s0, int64_t sens_s1, int32_t* iters_out) {
    if (!s) return fail(WLSQM_E_VALUE, "NULL solver");
    if (!s->ready) return fail(WLSQM_E_NOTREADY, "Solver is not in the ready state; prepare() must be called before solve()");
    if (s->ncases == 0) { if (iters_out) *iters_out = 0; return WLSQM_OK; }
    if (!s->hoods_dev.p) return fail(WLSQM_E_NOTREADY, "solve_hoods() needs the neighbour lists of prepare_hoods()");
    if (!f) return fail(WLSQM_E_VALUE, "f must not be NULL");
    int rc = use_device(s);
    if (rc) return rc;
    cudaStream_t st = s->stream;
    const long long n = s->ncases;
    const double* fd = f;
    long long fs0 = f_s0;
    if (!is_device_ptr(f)) {
        rc = s->hood_f.reserve((size_t)s->hood_points * 8);
        if (rc) return rc;
        rc = to_dense((double*)s->hood_f.p, f, s->hood_points, 1, f_s0, st);
        if (rc) return rc;
        fd = (const double*)s->hood_f.p;
        fs0 = 1;
    }
    // rows of the gathered fk get an EVEN pitch, so that the solve kernel can fetch them with bulk copies whatever nk is
    const long long kp = ((long long)s->maxnk + 1) & ~1ll;
    rc = s->hood_fk.reserve((size_t)n * kp * 8);
    if (rc) return rc;
    // (the indices were validated against [0, hood_points) by prepare_hoods; padding slots are not read)
    CU(gather_hoods(s, fd, fs0, 1, (int)kp, (double*)s->hood_fk.p, nullptr));
    return wlsqm_solver_solve(s, (const double*)s->hood_fk.p, kp, 1, fi, fi_s0, sens, sens_s0, sens_s1, iters_out);
}

// Several fields on one geometry (wlsqm_solve.cu, FieldsParams): fk given per case, or (hoods) per point through the
// neighbour lists of prepare_hoods (hf [nf][npoints], strides f_sf / f_s0).
static int solve_fields_core(wlsqm_solver_t* s, int64_t nf, bool hoods, const double* fk, int64_t fk_sf, int64_t fk_s0,
                             int64_t fk_s1, const double* hf, int64_t f_sf, int64_t f_s0, double* fi, int64_t fi_sf, int64_t fi_s0,
                             int32_t* iters_out) {
    if (!s) return fail(WLSQM_E_VALUE, "NULL solver");
    if (iters_out) *iters_out = 0;
    if (!s->ready) return fail(WLSQM_E_NOTREADY, "Solver is not in the ready state; prepare() must be called before solve()");
    if (nf < 0) return fail(WLSQM_E_VALUE, "nf must be >= 0, got %lld", (long long)nf);
    if (s->ngather > 0) return fail(WLSQM_E_VALUE, "the field solves do not support the fused result gather (wlsqm_solver_set_gather)");
    const long long n = s->ncases;
    if (nf == 0 || n == 0) return WLSQM_OK;
    if (hoods && !s->hoods_dev.p) return fail(WLSQM_E_NOTREADY, "solve_hoods_fields() needs the neighbour lists of prepare_hoods()");
    if ((hoods ? !hf : !fk) || !fi) return fail(WLSQM_E_VALUE, "fk (f) and fi must not be NULL");
    const int maxno = s->maxno, maxnk = s->maxnk;
    // the (field, case, slot) -> element map of fi must be injective: fields-outer or fields-inner rows
    if (!fields_layout_ok(nf, n, maxno, fi_sf, fi_s0))
        return fail(WLSQM_E_VALUE, "fi layout (field stride %lld, row stride %lld) maps two (field, case, slot) entries to one "
                    "element; use fields-outer (fi_sf >= (ncases-1)*fi_s0 + max no) or fields-inner (fi_sf >= max no, "
                    "fi_s0 >= (nf-1)*fi_sf + max no) rows", (long long)fi_sf, (long long)fi_s0);
    int rc = use_device(s);
    if (rc) return rc;
    cudaStream_t st = s->stream;
    const bool iter = s->algorithm == WLSQM_ALGO_ITERATIVE;
    const bool fk_dev = hoods ? true : is_device_ptr(fk) != 0, fi_dev = is_device_ptr(fi) != 0;
    if (!hoods && fk_dev && fi_dev) {
        // address span [lo, hi] of each strided array (element offsets)
        auto span = [](long long a, long long sa, long long b, long long sb, long long c, long long sc, long long& lo, long long& hi) {
            lo = hi = 0;
            for (long long t : {(a - 1) * sa, (b - 1) * sb, (c - 1) * sc}) (t < 0 ? lo : hi) += t;
        };
        long long klo, khi, ilo, ihi;
        span(nf, fk_sf, n, fk_s0, maxnk, fk_s1, klo, khi);
        span(nf, fi_sf, n, fi_s0, maxno, 1, ilo, ihi);
        if (ranges_overlap(fk + klo, (khi - klo + 1) * 8, fi + ilo, (ihi - ilo + 1) * 8))
            return fail(WLSQM_E_VALUE, "device fk overlaps device fi: the field solves write fi while other fields still read fk");
    }

    // ---- host arrays: staged whole (one dense device mirror per argument) -----------------------------------------------
    if (!hoods && !fk_dev) {
        if (fk_s1 != 1 && maxnk > 1) return fail(WLSQM_E_VALUE, "host fk must have unit stride on its last axis");
        rc = s->st_fk.reserve((size_t)nf * n * maxnk * 8);
        if (rc) return rc;
        for (long long j = 0; j < nf; ++j) {
            rc = to_dense((double*)s->st_fk.p + j * n * maxnk, fk + j * fk_sf, n, maxnk, fk_s0, st);
            if (rc) return rc;
        }
        fk = (const double*)s->st_fk.p; fk_sf = n * maxnk; fk_s0 = maxnk; fk_s1 = 1;
    }
    if (hoods && !is_device_ptr(hf)) {
        const long long np = s->hood_points;
        rc = s->hood_f.reserve((size_t)nf * np * 8);
        if (rc) return rc;
        for (long long j = 0; j < nf; ++j) {
            rc = to_dense((double*)s->hood_f.p + j * np, hf + j * f_sf, np, 1, f_s0, st);
            if (rc) return rc;
        }
        hf = (const double*)s->hood_f.p; f_sf = np; f_s0 = 1;
    }
    double* fi_use = fi;
    long long fi_sf_use = fi_sf, fi_s0_use = fi_s0;
    if (!fi_dev) {
        rc = s->st_fi.reserve((size_t)nf * n * maxno * 8);
        if (rc) return rc;
        for (long long j = 0; j < nf; ++j) {
            rc = to_dense((double*)s->st_fi.p + j * n * maxno, fi + j * fi_sf, n, maxno, fi_s0, st);
            if (rc) return rc;
        }
        fi_use = (double*)s->st_fi.p; fi_sf_use = n * maxno; fi_s0_use = maxno;
    }

    FieldsParams F{};
    SolveParams& P = F.P;
    solve_params(s, P);
    if (iter) CU(cudaMemsetAsync(s->iters_dev, 0, ((size_t)n + 1) * 4, st));   // per-case counts: maxima over the passes
    // gathered hood data: (fields of a pass, ncases, kp) with an EVEN row pitch kp, so that every row qualifies for bulk copies
    const long long kp = ((long long)maxnk + 1) & ~1ll;
    auto set_fk = [&](long long p0) {
        if (hoods) { P.fk = (const double*)s->hood_fk.p; P.fk_s0 = kp; P.fk_s1 = 1; F.fk_sf = n * kp; }
        else { P.fk = fk + p0 * fk_sf; P.fk_s0 = fk_s0; P.fk_s1 = fk_s1; F.fk_sf = fk_sf; }
    };
    const bool pack = pack_eligible(s);
    LaunchCfg L;
    // fields per pass: what one launch shape holds, spread evenly over the passes
    set_fk(0);
    F.nf = (int)std::min<int64_t>(nf, 1 << 20);
    rc = config_solve_fields(s, F, L, n, pack);
    if (rc) return rc;
    const long long passes = (nf + F.nf - 1) / F.nf, per_pass = (nf + passes - 1) / passes;
    if (hoods) {
        rc = s->hood_fk.reserve((size_t)per_pass * n * kp * 8);
        if (rc) return rc;
    }
    for (long long p0 = 0; p0 < nf; p0 += per_pass) {
        const int nfp = (int)std::min(per_pass, nf - p0);
        if (hoods) CU(gather_hoods(s, hf + p0 * f_sf, f_s0, 1, (int)kp, (double*)s->hood_fk.p, nullptr, nfp, f_sf, n * kp));
        set_fk(p0);
        F.fi = fi_use + p0 * fi_sf_use; F.fi_sf = fi_sf_use; F.fi_s0 = fi_s0_use;
        P.case_lo = 0; P.ncases = n;
        F.nf = nfp;
        auto config = [&](long long rows) {
            const int r = config_solve_fields(s, F, L, rows, pack);
            if (!r && F.nf != nfp) return fail(WLSQM_E_VALUE, "internal: %d fields per pass do not fit the launch shape", nfp);
            return r;
        };
        // (every field's row of the last case may end its array)
        if (pack) rc = launch_solve_split(P, false, config, [&] { return launch_solve_pack_fields(F, L.blocks, L.threads, L.smem, st); });
        else rc = launch_solve_split(P, s->last_nk_odd, config, [&] { return launch_solve_fields(s->dim, F, L.blocks, L.threads, L.smem, st); });
        if (rc) return rc;
    }
    // the solver's own solution copy is not written: interpolate / get_fi refuse until the next solve()
    s->fi_case_valid = false;
    if (!fi_dev) {
        for (long long j = 0; j < nf; ++j) {
            rc = from_dense(fi + j * fi_sf, fi_s0, (const double*)s->st_fi.p + j * n * maxno, maxno, n, maxno, st);
            if (rc) return rc;
        }
    }
    int32_t it = 0;
    if (iter) CU(cudaMemcpyAsync(&it, s->iters_dev, 4, cudaMemcpyDeviceToHost, st));
    if (iter || !fi_dev || !fk_dev) CU(cudaStreamSynchronize(st));
    if (iters_out) *iters_out = it;
    return WLSQM_OK;
}

int wlsqm_solver_solve_fields(wlsqm_solver_t* s, int64_t nf, const double* fk, int64_t fk_sf, int64_t fk_s0, int64_t fk_s1,
                              double* fi, int64_t fi_sf, int64_t fi_s0, int32_t* iters_out) {
    return solve_fields_core(s, nf, false, fk, fk_sf, fk_s0, fk_s1, nullptr, 0, 0, fi, fi_sf, fi_s0, iters_out);
}

int wlsqm_solver_solve_hoods_fields(wlsqm_solver_t* s, int64_t nf, const double* f, int64_t f_sf, int64_t f_s0, double* fi,
                                    int64_t fi_sf, int64_t fi_s0, int32_t* iters_out) {
    return solve_fields_core(s, nf, true, nullptr, 0, 0, 0, f, f_sf, f_s0, fi, fi_sf, fi_s0, iters_out);
}

// ---- export of the prepared operators (wlsqm_operator.cu) -------------------------------------------------------
// A guest answers with its host's operators and neighbour lists: everything below reads the lender's state.
static int opx_check(wlsqm_solver_t* s, int nops, const double* coeffs, bool hoods) {
    if (!s) return fail(WLSQM_E_VALUE, "NULL solver");
    const wlsqm_solver* r = s->lender ? s->lender : s;
    if (!r->ready) return fail(WLSQM_E_NOTREADY, "Solver is not in the ready state; prepare() must be called first");
    if (hoods && !r->hoods_current)
        return fail(WLSQM_E_NOTREADY, "the global operator needs the neighbour lists of prepare_hoods() as the last prepare");
    if (nops < 1 || nops > WLSQM_MAXNO) return fail(WLSQM_E_VALUE, "nops must be 1..%d, got %d", WLSQM_MAXNO, nops);
    if (!coeffs) return fail(WLSQM_E_VALUE, "coeffs must not be NULL");
    for (long long t = 0; t < (long long)nops * s->maxno; ++t)
        if (!std::isfinite(coeffs[t])) return fail(WLSQM_E_VALUE, "coefficients must be finite (entry %lld)", t);
    return use_device(s);
}

static int opx_center(const wlsqm_solver* s, int64_t center) {
    const wlsqm_solver* r = s->lender ? s->lender : s;
    if (center != -1 && (center < 0 || center + s->ncases > r->hood_points))
        return fail(WLSQM_E_VALUE, "center must be -1 (no folding) or 0 <= center, center + ncases <= npoints = %lld; got %lld",
                    (long long)r->hood_points, (long long)center);
    return WLSQM_OK;
}

// W [nops][ncases][maxnk], K [nops][ncases][maxno] (or NULL), kf [nops][ncases] (or NULL): device pointers
static int opx_stencils(wlsqm_solver_t* s, int nops, const double* coeffs, double* W, double* K, double* kf) {
    const wlsqm_solver* r = s->lender ? s->lender : s;
    if (s->lender) CU(order_streams(r->stream, s->stream));   // the host's prepare may still be in flight
    const int maxno = s->maxno;
    int rc = s->opx_coef.reserve((size_t)nops * maxno * 8);
    if (rc) return rc;
    CU(cudaMemcpyAsync(s->opx_coef.p, coeffs, (size_t)nops * maxno * 8, cudaMemcpyHostToDevice, s->stream));
    StencilParams P{};
    P.meta = r->dmeta; P.uni = r->uni; P.geom_uniform = r->geom_uniform ? 1 : 0; P.op_stride = r->op_stride;
    P.ncases = s->ncases; P.op = r->op; P.coef = (const double*)s->opx_coef.p;
    P.nops = nops; P.maxnk = s->maxnk; P.maxno = maxno; P.W = W; P.K = K; P.kf = kf;
    // the ring of solve_kernel: two stages of the largest block, 16 warps per SM for blocks of 3 KB and more
    P.stage_doubles = std::max(2, even(s->maxnq * s->maxnr));
    P.ring_off = (nops * maxno + nops + 15) & ~15;
    const size_t stage_bytes = (size_t)P.stage_doubles * 8;
    int S = 2, warps = stage_bytes >= 3072 ? 16 : 32;
    size_t smem = 0;
    for (;;) {
        smem = (size_t)P.ring_off * 8 + (size_t)warps * S * (stage_bytes + 8);
        if (smem <= SMEM_PER_CTA) break;
        if (warps > 4) --warps;
        else if (S > 1) --S;
        else if (warps > 1) --warps;
        else return fail(WLSQM_E_VALUE, "operator block too large for shared memory (%zu bytes)", stage_bytes);
    }
    P.stages = S;
    P.bar_off_bytes = P.ring_off * 8 + warps * S * P.stage_doubles * 8;
    const int blocks = grid_blocks(s, smem, warps, stage_bytes >= 3072 ? 16 : 32, s->ncases);
    CU(launch_stencils(P, blocks, warps * 32, smem, s->stream));
    return WLSQM_OK;
}

// a device view of an output: the caller's pointer, or a staging buffer copied back by opx_copy_out
static int opx_out(void* p, size_t bytes, DevBuf& stage, void** dev) {
    *dev = p;
    if (!p || is_device_ptr(p)) return WLSQM_OK;
    int rc = stage.reserve(bytes);
    if (rc) return rc;
    *dev = stage.p;
    return WLSQM_OK;
}
static int opx_copy_out(void* p, const void* dev, size_t bytes, cudaStream_t st) {
    if (p && p != dev && bytes) CU(cudaMemcpyAsync(p, dev, bytes, cudaMemcpyDeviceToHost, st));
    return WLSQM_OK;
}

// count pass + scan: rp [n + 1] (device), nnz on the host.  Rows are the cases (row_case == nullptr, n == ncases) or
// queries with their case index (device int64 [n], the interpolation operators)
static int opx_pattern(wlsqm_solver_t* s, int64_t center, long long n, const long long* row_case, DevBuf& cnt, DevBuf& rp,
                       CsrParams& P, long long* nnz) {
    const wlsqm_solver* r = s->lender ? s->lender : s;
    if (s->lender) CU(order_streams(r->stream, s->stream));
    if (n >= (1LL << 31) - 1) return fail(WLSQM_E_VALUE, "the global operator supports up to 2^31 - 2 rows");
    if ((size_t)CSR_BYTES_PER_NK * r->maxnk > CSR_SMEM_MAX)
        return fail(WLSQM_E_VALUE, "the global operator supports up to %zu neighbours per case, got %d",
                    CSR_SMEM_MAX / CSR_BYTES_PER_NK, r->maxnk);
    int rc = cnt.reserve((size_t)(n + 1) * 8);
    if (!rc) rc = rp.reserve((size_t)(n + 1) * 8);
    if (rc) return rc;
    P.meta = r->dmeta; P.uni = r->uni; P.ncases = n; P.row_case = row_case; P.nmodels = s->ncases;
    P.hoods = (const int32_t*)r->hoods_dev.p; P.hoods_s0 = r->maxnk; P.maxnk = r->maxnk;
    P.center = center;
    P.cnt = (long long*)cnt.p;
    CU(cudaMemsetAsync((long long*)cnt.p + n, 0, 8, s->stream));
    CU(launch_csr_count(P, s->stream));
    size_t tb = 0;
    CU(csr_scan((long long*)cnt.p, (long long*)rp.p, n + 1, nullptr, &tb, s->stream));
    DevBuf tmp;
    rc = tmp.reserve(tb + 16);
    if (rc) return rc;
    tb += 16;
    long long total = 0;
    cudaError_t e = csr_scan((long long*)cnt.p, (long long*)rp.p, n + 1, tmp.p, &tb, s->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&total, (long long*)rp.p + n, 8, cudaMemcpyDeviceToHost, s->stream);
    const cudaError_t e2 = cudaStreamSynchronize(s->stream);
    tmp.release();
    if (e == cudaSuccess) e = e2;
    if (e != cudaSuccess) return fail(WLSQM_E_CUDA, "operator pattern: %s", cudaGetErrorString(e));
    P.rp = (const long long*)rp.p;
    P.nnz = total;
    *nnz = total;
    return WLSQM_OK;
}

int wlsqm_solver_stencils(wlsqm_solver_t* s, int nops, const double* coeffs, double* W, double* K) {
    int rc = opx_check(s, nops, coeffs, false);
    if (rc) return rc;
    if (!W) return fail(WLSQM_E_VALUE, "W must not be NULL");
    if (s->ncases == 0) return WLSQM_OK;
    const size_t wb = (size_t)nops * s->ncases * s->maxnk * 8, kb = (size_t)nops * s->ncases * s->maxno * 8;
    DevBuf sw, sk;
    void *Wd, *Kd;
    rc = opx_out(W, wb, sw, &Wd);
    if (!rc) rc = opx_out(K, kb, sk, &Kd);
    if (!rc) rc = opx_stencils(s, nops, coeffs, (double*)Wd, (double*)Kd, nullptr);
    if (!rc) rc = opx_copy_out(W, Wd, wb, s->stream);
    if (!rc && K) rc = opx_copy_out(K, Kd, kb, s->stream);
    if (sw.p || sk.p) {
        const cudaError_t e = cudaStreamSynchronize(s->stream);
        sw.release(); sk.release();
        if (!rc && e != cudaSuccess) return fail(WLSQM_E_CUDA, "stencils: %s", cudaGetErrorString(e));
    }
    return rc;
}

int wlsqm_solver_operator_nnz(wlsqm_solver_t* s, int64_t center, int64_t* nnz) {
    if (!nnz) return fail(WLSQM_E_VALUE, "nnz must not be NULL");
    *nnz = 0;
    if (!s) return fail(WLSQM_E_VALUE, "NULL solver");
    const wlsqm_solver* r = s->lender ? s->lender : s;
    if (!r->ready) return fail(WLSQM_E_NOTREADY, "Solver is not in the ready state; prepare() must be called first");
    if (!r->hoods_current)
        return fail(WLSQM_E_NOTREADY, "the global operator needs the neighbour lists of prepare_hoods() as the last prepare");
    int rc = opx_center(s, center);
    if (rc) return rc;
    if (s->ncases == 0) return WLSQM_OK;
    rc = use_device(s);
    if (rc) return rc;
    DevBuf cnt, rp;
    CsrParams P{};
    long long total = 0;
    rc = opx_pattern(s, center, s->ncases, nullptr, cnt, rp, P, &total);
    cudaStreamSynchronize(s->stream);
    cnt.release(); rp.release();
    if (rc) return rc;
    *nnz = total;
    return WLSQM_OK;
}

int wlsqm_solver_operator_csr(wlsqm_solver_t* s, int nops, const double* coeffs, int64_t center, int index_bits, void* rowptr,
                              void* col, double* values, double* K) {
    int rc = opx_check(s, nops, coeffs, true);
    if (rc) return rc;
    rc = opx_center(s, center);
    if (rc) return rc;
    if (index_bits != 32 && index_bits != 64) return fail(WLSQM_E_VALUE, "index_bits must be 32 or 64, got %d", index_bits);
    if (!rowptr) return fail(WLSQM_E_VALUE, "rowptr must not be NULL");
    const long long n = s->ncases;
    const size_t ib = index_bits / 8;
    if (n == 0) {
        const long long z = 0;
        if (is_device_ptr(rowptr)) CU(cudaMemcpy(rowptr, &z, ib, cudaMemcpyHostToDevice));
        else memcpy(rowptr, &z, ib);
        return WLSQM_OK;
    }
    DevBuf cnt, rp, wtmp, kf, s_rp, s_col, s_val, s_k;
    struct Release {     // every scratch block goes back once the stream is idle
        wlsqm_solver_t* s; DevBuf* b[8];
        ~Release() { cudaStreamSynchronize(s->stream); for (DevBuf* d : b) d->release(); }
    } release{s, {&cnt, &rp, &wtmp, &kf, &s_rp, &s_col, &s_val, &s_k}};
    CsrParams P{};
    long long nnz = 0;
    rc = opx_pattern(s, center, n, nullptr, cnt, rp, P, &nnz);
    if (rc) return rc;
    if (index_bits == 32 && nnz >= (1LL << 31))
        return fail(WLSQM_E_VALUE, "nnz = %lld does not fit 32-bit indices; use index_bits = 64", nnz);
    if (nnz > 0 && (!col || !values)) return fail(WLSQM_E_VALUE, "col and values must not be NULL");
    rc = wtmp.reserve((size_t)nops * n * std::max(s->maxnk, 1) * 8);
    if (!rc && center >= 0) rc = kf.reserve((size_t)nops * n * 8);
    if (rc) return rc;
    const size_t rb = (size_t)(n + 1) * ib, cb = (size_t)nnz * ib, vb = (size_t)nops * nnz * 8, kb = (size_t)nops * n * s->maxno * 8;
    void *rpd, *cd, *vd, *kd;
    rc = opx_out(rowptr, rb, s_rp, &rpd);
    if (!rc) rc = opx_out(nnz ? col : nullptr, cb, s_col, &cd);
    if (!rc) rc = opx_out(nnz ? values : nullptr, vb, s_val, &vd);
    if (!rc) rc = opx_out(K, kb, s_k, &kd);
    if (!rc) rc = opx_stencils(s, nops, coeffs, (double*)wtmp.p, (double*)kd, center >= 0 ? (double*)kf.p : nullptr);
    if (rc) return rc;
    P.W = (const double*)wtmp.p; P.kf = (const double*)kf.p; P.nops = nops;
    P.rowptr = rpd; P.col = cd; P.values = (double*)vd;
    CU(launch_csr_fill(P, index_bits, s->stream));
    rc = opx_copy_out(rowptr, rpd, rb, s->stream);
    if (!rc && nnz) rc = opx_copy_out(col, cd, cb, s->stream);
    if (!rc && nnz) rc = opx_copy_out(values, vd, vb, s->stream);
    if (!rc && K) rc = opx_copy_out(K, kd, kb, s->stream);
    if (rc) return rc;
    CU(cudaStreamSynchronize(s->stream));
    return WLSQM_OK;
}

// ---- interpolation operators: rows at query points (wlsqm_operator.cu) ----------------------------------------
// a device view of the case indices I [nx] (int64): the caller's array, or the solver's staging copy
static int opx_index(wlsqm_solver_t* s, const int64_t* I, long long nx, const long long** Id) {
    if (!I) return fail(WLSQM_E_VALUE, "I must not be NULL");
    if (nx >= (1LL << 31) - 1) return fail(WLSQM_E_VALUE, "the interpolation operators support up to 2^31 - 2 queries");
    if (is_device_ptr(I)) { *Id = (const long long*)I; return WLSQM_OK; }
    int rc = s->st_I.reserve((size_t)nx * 8);
    if (!rc) rc = stage_in(s->device, (double*)s->st_I.p, reinterpret_cast<const double*>(I), nx, 1, 1, s->stream);   // (8-byte items)
    if (rc) return rc;
    *Id = (const long long*)s->st_I.p;
    return WLSQM_OK;
}
// ... and of the query points x [nx][dim] (row pitch x_s0)
static int opx_points(wlsqm_solver_t* s, const double* x, int64_t x_s0, long long nx, const double** xd, long long* xs) {
    if (!x) return fail(WLSQM_E_VALUE, "x must not be NULL");
    if (is_device_ptr(x)) { *xd = x; *xs = x_s0; return WLSQM_OK; }
    int rc = s->st_x.reserve((size_t)nx * s->dim * 8);
    if (!rc) rc = stage_in(s->device, (double*)s->st_x.p, x, nx, s->dim, x_s0, s->stream);
    if (rc) return rc;
    *xd = (const double*)s->st_x.p; *xs = s->dim;
    return WLSQM_OK;
}

// W [nops][nx][maxnk], K [nops][nx][maxno] (or NULL), kf [nops][nx] (or NULL) of the queries: device pointers.
// Continuous mode: the nx rows are pairs, row p at query row_query[p] with its coefficient rows scaled by row_scale[p].
static int opx_interp(wlsqm_solver_t* s, const double* xd, long long xs, const long long* Id, long long nx, int nops,
                      const double* coeffs, double* W, double* K, double* kf, const int* row_query = nullptr,
                      const double* row_scale = nullptr) {
    const wlsqm_solver* r = s->lender ? s->lender : s;
    if (s->lender) CU(order_streams(r->stream, s->stream));   // the host's prepare may still be in flight
    const int maxno = s->maxno;
    // runs of equal I among the queries
    int rc = s->opx_runs.reserve(((size_t)7 * nx + 1) * sizeof(int));
    if (rc) return rc;
    int* rb = (int*)s->opx_runs.p;
    InterpRuns R{rb, rb + nx, rb + 2 * nx, rb + 3 * nx, rb + 4 * nx, rb + 5 * nx, rb + 6 * nx, rb + 7 * nx};
    size_t tb = 0;
    CU(interp_runs(Id, nx, s->ncases, R, nullptr, &tb, s->stream));
    rc = s->opx_tmp.reserve(tb + 16);
    if (rc) return rc;
    tb = s->opx_tmp.cap;
    CU(interp_runs(Id, nx, s->ncases, R, s->opx_tmp.p, &tb, s->stream));
    rc = s->opx_coef.reserve((size_t)nops * maxno * 8);
    if (rc) return rc;
    CU(cudaMemcpyAsync(s->opx_coef.p, coeffs, (size_t)nops * maxno * 8, cudaMemcpyHostToDevice, s->stream));
    InterpStencilParams P{};
    P.meta = r->dmeta; P.uni = r->uni; P.geom_uniform = r->geom_uniform ? 1 : 0; P.op_stride = r->op_stride;
    P.nmodels = s->ncases; P.op = r->op; P.xi = r->xi_dev; P.x = xd; P.x_s0 = xs; P.dim = s->dim; P.nx = nx;
    P.run_case = R.run_case; P.run_len = R.run_len; P.run_off = R.run_off; P.nruns = R.nruns; P.perm = R.perm;
    P.coef = (const double*)s->opx_coef.p; P.nops = nops; P.maxnk = s->maxnk; P.maxno = maxno;
    P.W = W; P.K = K; P.kf = kf; P.row_query = row_query; P.row_scale = row_scale;
    // the ring of stencil_kernel, plus per warp the coefficient rows of one query (all nops operators, or fewer per pass
    // when shared memory is short) and its Taylor terms
    P.stage_doubles = std::max(2, even(s->maxnq * s->maxnr));
    P.ring_off = (nops * maxno + nops + (maxno + 3) / 4 + 15) & ~15;
    const size_t stage_bytes = (size_t)P.stage_doubles * 8;
    int S = 2, warps = stage_bytes >= 3072 ? 16 : 32, opc = nops, cqd = 0;
    size_t smem = 0;
    for (;;) {
        cqd = even(opc * maxno + opc + 15);
        smem = (size_t)P.ring_off * 8 + (size_t)warps * S * (stage_bytes + 8) + (size_t)warps * cqd * 8;
        if (smem <= SMEM_PER_CTA) break;
        if (warps > 8) --warps;
        else if (opc > 1) opc = (opc + 1) / 2;
        else if (warps > 4) --warps;
        else if (S > 1) --S;
        else if (warps > 1) --warps;
        else return fail(WLSQM_E_VALUE, "operator block too large for shared memory (%zu bytes)", stage_bytes);
    }
    P.stages = S; P.opc = opc; P.cq_doubles = cqd;
    P.cq_off = P.ring_off + warps * S * P.stage_doubles;
    P.bar_off_bytes = (P.cq_off + warps * cqd) * 8;
    const int blocks = grid_blocks(s, smem, warps, stage_bytes >= 3072 ? 16 : 32, nx);   // (there are at most nx runs)
    CU(launch_interp_stencils(P, blocks, warps * 32, smem, s->stream));
    return WLSQM_OK;
}

int wlsqm_solver_interp_stencils(wlsqm_solver_t* s, const double* x, int64_t x_s0, const int64_t* I, int64_t nx, int nops,
                                 const double* coeffs, double* W, double* K) {
    int rc = opx_check(s, nops, coeffs, false);
    if (rc) return rc;
    if (nx < 0) return fail(WLSQM_E_VALUE, "nx must be >= 0, got %lld", (long long)nx);
    if (nx == 0) return WLSQM_OK;
    if (!W) return fail(WLSQM_E_VALUE, "W must not be NULL");
    const double* xd;
    long long xs;
    const long long* Id;
    rc = opx_index(s, I, nx, &Id);
    if (!rc) rc = opx_points(s, x, x_s0, nx, &xd, &xs);
    if (rc) return rc;
    const size_t wb = (size_t)nops * nx * s->maxnk * 8, kb = (size_t)nops * nx * s->maxno * 8;
    DevBuf sw, sk;
    void *Wd, *Kd;
    rc = opx_out(W, wb, sw, &Wd);
    if (!rc) rc = opx_out(K, kb, sk, &Kd);
    if (!rc) rc = opx_interp(s, xd, xs, Id, nx, nops, coeffs, (double*)Wd, (double*)Kd, nullptr);
    if (!rc) rc = opx_copy_out(W, Wd, wb, s->stream);
    if (!rc && K) rc = opx_copy_out(K, Kd, kb, s->stream);
    if (sw.p || sk.p || xd != x || (const void*)Id != (const void*)I) {
        const cudaError_t e = cudaStreamSynchronize(s->stream);
        sw.release(); sk.release();
        if (!rc && e != cudaSuccess) return fail(WLSQM_E_CUDA, "interp_stencils: %s", cudaGetErrorString(e));
    }
    return rc;
}

int wlsqm_solver_interp_operator_nnz(wlsqm_solver_t* s, const int64_t* I, int64_t nx, int64_t center, int64_t* nnz) {
    if (!nnz) return fail(WLSQM_E_VALUE, "nnz must not be NULL");
    *nnz = 0;
    if (!s) return fail(WLSQM_E_VALUE, "NULL solver");
    const wlsqm_solver* r = s->lender ? s->lender : s;
    if (!r->ready) return fail(WLSQM_E_NOTREADY, "Solver is not in the ready state; prepare() must be called first");
    if (!r->hoods_current)
        return fail(WLSQM_E_NOTREADY, "the global operator needs the neighbour lists of prepare_hoods() as the last prepare");
    int rc = opx_center(s, center);
    if (rc) return rc;
    if (nx < 0) return fail(WLSQM_E_VALUE, "nx must be >= 0, got %lld", (long long)nx);
    if (nx == 0) return WLSQM_OK;
    rc = use_device(s);
    if (rc) return rc;
    const long long* Id;
    rc = opx_index(s, I, nx, &Id);
    if (rc) return rc;
    DevBuf cnt, rp;
    CsrParams P{};
    long long total = 0;
    rc = opx_pattern(s, center, nx, Id, cnt, rp, P, &total);
    cudaStreamSynchronize(s->stream);
    cnt.release(); rp.release();
    if (rc) return rc;
    *nnz = total;
    return WLSQM_OK;
}

int wlsqm_solver_interp_operator_csr(wlsqm_solver_t* s, const double* x, int64_t x_s0, const int64_t* I, int64_t nx, int nops,
                                     const double* coeffs, int64_t center, int index_bits, void* rowptr, void* col,
                                     double* values, double* K) {
    int rc = opx_check(s, nops, coeffs, true);
    if (rc) return rc;
    rc = opx_center(s, center);
    if (rc) return rc;
    if (index_bits != 32 && index_bits != 64) return fail(WLSQM_E_VALUE, "index_bits must be 32 or 64, got %d", index_bits);
    if (!rowptr) return fail(WLSQM_E_VALUE, "rowptr must not be NULL");
    if (nx < 0) return fail(WLSQM_E_VALUE, "nx must be >= 0, got %lld", (long long)nx);
    const size_t ib = index_bits / 8;
    if (nx == 0) {
        const long long z = 0;
        if (is_device_ptr(rowptr)) CU(cudaMemcpy(rowptr, &z, ib, cudaMemcpyHostToDevice));
        else memcpy(rowptr, &z, ib);
        return WLSQM_OK;
    }
    const double* xd;
    long long xs;
    const long long* Id;
    rc = opx_index(s, I, nx, &Id);
    if (!rc) rc = opx_points(s, x, x_s0, nx, &xd, &xs);
    if (rc) return rc;
    DevBuf cnt, rp, wtmp, kf, s_rp, s_col, s_val, s_k;
    struct Release {     // every scratch block goes back once the stream is idle
        wlsqm_solver_t* s; DevBuf* b[8];
        ~Release() { cudaStreamSynchronize(s->stream); for (DevBuf* d : b) d->release(); }
    } release{s, {&cnt, &rp, &wtmp, &kf, &s_rp, &s_col, &s_val, &s_k}};
    CsrParams P{};
    long long nnz = 0;
    rc = opx_pattern(s, center, nx, Id, cnt, rp, P, &nnz);
    if (rc) return rc;
    if (index_bits == 32 && nnz >= (1LL << 31))
        return fail(WLSQM_E_VALUE, "nnz = %lld does not fit 32-bit indices; use index_bits = 64", nnz);
    if (nnz > 0 && (!col || !values)) return fail(WLSQM_E_VALUE, "col and values must not be NULL");
    rc = wtmp.reserve((size_t)nops * nx * std::max(s->maxnk, 1) * 8);
    if (!rc && center >= 0) rc = kf.reserve((size_t)nops * nx * 8);
    if (rc) return rc;
    const size_t rb = (size_t)(nx + 1) * ib, cb = (size_t)nnz * ib, vb = (size_t)nops * nnz * 8, kb = (size_t)nops * nx * s->maxno * 8;
    void *rpd, *cd, *vd, *kd;
    rc = opx_out(rowptr, rb, s_rp, &rpd);
    if (!rc) rc = opx_out(nnz ? col : nullptr, cb, s_col, &cd);
    if (!rc) rc = opx_out(nnz ? values : nullptr, vb, s_val, &vd);
    if (!rc) rc = opx_out(K, kb, s_k, &kd);
    if (!rc) rc = opx_interp(s, xd, xs, Id, nx, nops, coeffs, (double*)wtmp.p, (double*)kd, center >= 0 ? (double*)kf.p : nullptr);
    if (rc) return rc;
    P.W = (const double*)wtmp.p; P.kf = (const double*)kf.p; P.nops = nops;
    P.rowptr = rpd; P.col = cd; P.values = (double*)vd;
    CU(launch_csr_fill(P, index_bits, s->stream));
    rc = opx_copy_out(rowptr, rpd, rb, s->stream);
    if (!rc && nnz) rc = opx_copy_out(col, cd, cb, s->stream);
    if (!rc && nnz) rc = opx_copy_out(values, vd, vb, s->stream);
    if (!rc && K) rc = opx_copy_out(K, kd, kb, s->stream);
    if (rc) return rc;
    CU(cudaStreamSynchronize(s->stream));
    return WLSQM_OK;
}

int wlsqm_solver_index_models(wlsqm_solver_t* s) {
    if (!s) return fail(WLSQM_E_VALUE, "NULL solver");
    if (!s->ready) return fail(WLSQM_E_NOTREADY, "Solver is not in the ready state; prepare() must be called before prep_interpolate()");
    if (s->models_grid || s->ncases == 0) return WLSQM_OK;
    int rc = use_device(s);
    if (rc) return rc;
    CU(cudaStreamSynchronize(s->stream));
    return wlsqm_grid_create(s->dim, s->ncases, s->xi_dev, s->dim, s->device, &s->models_grid);
}

int wlsqm_solver_nearest_models(wlsqm_solver_t* s, const double* x, int64_t x_s0, int64_t nx, int64_t* I_out) {
    if (!s) return fail(WLSQM_E_VALUE, "NULL solver");
    if (!s->models_grid) return fail(WLSQM_E_NOTREADY, "Points xi have not been indexed; prep_interpolate() must be called before interpolate()");
    if (nx == 0) return WLSQM_OK;
    if (!x || !I_out) return fail(WLSQM_E_VALUE, "NULL argument");
    return wlsqm_grid_knn(s->models_grid, x, x_s0, nx, 1, 0, nullptr, I_out, nullptr);
}

int wlsqm_solver_interpolate_continuous(wlsqm_solver_t* s, const double* x, int64_t x_s0, int64_t nx, double r, int diff,
                                        double* out) {
    if (!s) return fail(WLSQM_E_VALUE, "NULL solver");
    if (!s->ready) return fail(WLSQM_E_NOTREADY, "Solver is not in the ready state; prepare() must be called first");
    if (!s->models_grid) return fail(WLSQM_E_NOTREADY, "Points xi have not been indexed; prep_interpolate() must be called before interpolate()");
    if (nx == 0) return WLSQM_OK;
    if (!x || !out) return fail(WLSQM_E_VALUE, "x and out must not be NULL");
    if (!(r > 0.0)) return fail(WLSQM_E_VALUE, "r must be positive");
    if (!s->fi_case_valid) return fail(WLSQM_E_NOTREADY, "the solver keeps no copy of the solution (wlsqm_solver_keep_solution(s, 0)); solve() again with the copy enabled");
    const int size = number_of_dofs(s->dim, 4);
    if (diff < 0 || diff >= size) return fail(WLSQM_E_VALUE, "invalid diff %d", diff);
    int rc = use_device(s);
    if (rc) return rc;
    cudaStream_t st = s->stream;
    const bool x_dev = is_device_ptr(x), out_dev = is_device_ptr(out);
    InterpParams P{};
    P.dim = s->dim; P.nx = nx; P.diff = diff;
    P.xi = s->xi_dev; P.xi_s0 = s->dim; P.fi = s->fi_case; P.fi_s0 = s->maxno;
    P.order = s->dorder; P.order_uniform = s->uni.order;
    if (x_dev) { P.x = x; P.x_s0 = x_s0; }
    else {
        rc = s->st_x.reserve((size_t)nx * s->dim * 8);
        if (rc) return rc;
        rc = stage_in(s->device, (double*)s->st_x.p, x, nx, s->dim, x_s0, st);
        if (rc) return rc;
        P.x = (const double*)s->st_x.p; P.x_s0 = s->dim;
    }
    if (out_dev) P.out = out;
    else {
        rc = s->st_out.reserve((size_t)nx * 8);
        if (rc) return rc;
        P.out = (double*)s->st_out.p;
    }
    P.out_s0 = 1;
    CU(launch_interpolate_continuous(P, grid_view(s->models_grid), r, st));
    if (!out_dev) CU(cudaMemcpyAsync(out, s->st_out.p, (size_t)nx * 8, cudaMemcpyDeviceToHost, st));
    if (!x_dev || !out_dev) CU(cudaStreamSynchronize(st));
    return WLSQM_OK;
}

// ---- continuous-mode interpolation operators (wlsqm_operator.cu) --------------------------------------------------
// The pairs (q, m) of the models within r come from the ball search over the solver's own model grid (the grid of
// interpolate(mode='continuous')); operators and neighbour lists are the lender's.
static int cont_check(wlsqm_solver_t* s, long long nx, double r) {
    if (!s) return fail(WLSQM_E_VALUE, "NULL solver");
    const wlsqm_solver* rt = s->lender ? s->lender : s;
    if (!rt->ready) return fail(WLSQM_E_NOTREADY, "Solver is not in the ready state; prepare() must be called first");
    if (!s->models_grid) return fail(WLSQM_E_NOTREADY, "Points xi have not been indexed; prep_interpolate() must be called before interpolate()");
    if (!(r > 0.0)) return fail(WLSQM_E_VALUE, "r must be positive");
    if (nx < 0) return fail(WLSQM_E_VALUE, "nx must be >= 0, got %lld", nx);
    if (nx >= (1LL << 31) - 1) return fail(WLSQM_E_VALUE, "the interpolation operators support up to 2^31 - 2 queries");
    return WLSQM_OK;
}

// pp: pair_ptr [nx + 1] (device); models: J [npairs] (int64, device), the query pq and the weight alpha of each pair
struct ContPairs {
    DevBuf pp, j32, pq, alpha;
    long long npairs = 0;
};

// pair_ptr of the queries xd (device, row pitch xs); the ball search returns when its outputs are written
static int cont_count(wlsqm_solver_t* s, const double* xd, long long xs, long long nx, double r, ContPairs& C) {
    int rc = C.pp.reserve((size_t)(nx + 1) * 8);
    if (rc) return rc;
    CU(cudaStreamSynchronize(s->stream));     // staged queries, earlier work on the solver's stream
    int64_t np = 0;
    rc = wlsqm_grid_ball_count(s->models_grid, xd, xs, nx, &r, 0, 0, 0, (int64_t*)C.pp.p, nullptr, &np);
    if (rc) return rc;
    C.npairs = np;
    return WLSQM_OK;
}

// the models of the pairs (ascending per query) -> Jd [npairs], and their queries and weights
static int cont_models(wlsqm_solver_t* s, const double* xd, long long xs, long long nx, double r, ContPairs& C, long long* Jd) {
    const long long np = C.npairs;
    if (np >= (1LL << 31) - 1) return fail(WLSQM_E_VALUE, "%lld pairs in one call exceed 2^31 - 2: split the queries", np);
    int rc = C.j32.reserve((size_t)std::max(np, 1LL) * 4);
    if (!rc) rc = C.pq.reserve((size_t)std::max(np, 1LL) * 4);
    if (!rc) rc = C.alpha.reserve((size_t)std::max(np, 1LL) * 8);
    if (rc) return rc;
    rc = wlsqm_grid_ball_csr(s->models_grid, xd, xs, nx, &r, 0, 0, 0, WLSQM_BALL_BY_INDEX, (const int64_t*)C.pp.p,
                             (int32_t*)C.j32.p);
    if (rc) return rc;
    CU(launch_cont_weights(xd, xs, s->dim, s->xi_dev, nx, r, (const long long*)C.pp.p, (const int32_t*)C.j32.p, Jd,
                           (int*)C.pq.p, (double*)C.alpha.p, s->stream));
    return WLSQM_OK;
}

// the caller's pair_ptr must be the one of wlsqm_solver_interp_continuous_count for the same x and r
static int cont_same_ptr(wlsqm_solver_t* s, const int64_t* pair_ptr, const ContPairs& C, long long nx) {
    DevBuf staged, flag;
    const long long* pd = (const long long*)pair_ptr;
    int rc = flag.reserve(4);
    if (!rc && !is_device_ptr(pair_ptr)) {
        rc = staged.reserve((size_t)(nx + 1) * 8);
        if (!rc) pd = (const long long*)staged.p;
    }
    if (rc) return rc;
    int bad = 0;
    cudaError_t e = cudaSuccess;
    if (pd != (const long long*)pair_ptr) e = cudaMemcpyAsync(staged.p, pair_ptr, (size_t)(nx + 1) * 8, cudaMemcpyHostToDevice, s->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(flag.p, 0, 4, s->stream);
    if (e == cudaSuccess) e = launch_ptr_mismatch(pd, (const long long*)C.pp.p, nx + 1, (int*)flag.p, s->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&bad, flag.p, 4, cudaMemcpyDeviceToHost, s->stream);
    const cudaError_t e2 = cudaStreamSynchronize(s->stream);
    staged.release(); flag.release();
    if (e == cudaSuccess) e = e2;
    if (e != cudaSuccess) return fail(WLSQM_E_CUDA, "pair_ptr: %s", cudaGetErrorString(e));
    if (bad) return fail(WLSQM_E_VALUE, "pair_ptr does not match the pairs of x and r (wlsqm_solver_interp_continuous_count)");
    return WLSQM_OK;
}

// The CSR pattern over the pairs and its fill.  Rows of at most row_cap candidate slots (max nk + 1 per pair) are merged
// by one warp in shared memory; longer rows by the sort route, over chunks of consecutive queries of at most
// WLSQM_CONT_CHUNK_SLOTS slots (default 2^26; a single longer row is one chunk), so that the scratch stays bounded and no
// call is refused for its total size.  WLSQM_CONT_ROW_CAP (default 2048, rounded up to a power of two; 0: every row
// takes the sort route) sets row_cap.
struct ContPattern {
    DevBuf cnt, rp, seg, keys, cand, keys_s, cand_s, head, hpos, tmp;
    std::vector<long long> hp;      // pair_ptr on the host
    long long chunk_slots = 0;
};

// the chunks of the sort route: each [q0, q1) starts at a long row; fn(q0, q1) runs one
static int cont_chunks(const ContCsrParams& P, const ContPattern& B, const std::function<int(long long, long long)>& fn) {
    const long long nx = P.nx, L = P.L;
    long long q0 = 0;
    for (;;) {
        while (q0 < nx && (B.hp[q0 + 1] - B.hp[q0]) * L <= P.row_cap) ++q0;
        if (q0 >= nx) return WLSQM_OK;
        long long q1 = q0 + 1;
        while (q1 < nx && (B.hp[q1 + 1] - B.hp[q0]) * L <= B.chunk_slots) ++q1;
        const int rc = fn(q0, q1);
        if (rc) return rc;
        q0 = q1;
    }
}

static int cont_chunk_run(wlsqm_solver_t* s, ContCsrParams& P, ContPattern& B, long long q0, long long q1, bool fill,
                          int index_bits) {
    P.q0 = q0; P.q1 = q1; P.slot0 = B.hp[q0] * P.L; P.nslots = (B.hp[q1] - B.hp[q0]) * P.L;
    CU(cont_long_rows(P, fill, index_bits, B.tmp.p, &B.tmp.cap, s->stream));
    return WLSQM_OK;
}

// count pass: the row counts and their scan (B.rp, nnz on the host); P is ready for the fill afterwards
static int cont_pattern(wlsqm_solver_t* s, const ContPairs& C, long long nx, int64_t center, const long long* Jd,
                        ContPattern& B, ContCsrParams& P, long long* nnz) {
    const wlsqm_solver* r = s->lender ? s->lender : s;
    if (s->lender) CU(order_streams(r->stream, s->stream));
    if (r->hood_points > (long long)CONT_NO_COLUMN - 1)
        return fail(WLSQM_E_VALUE, "the continuous-mode operator supports up to 2^32 - 2 points, got %lld", r->hood_points);
    const long long L = r->maxnk + 1;
    B.hp.assign(nx + 1, 0);
    CU(cudaMemcpyAsync(B.hp.data(), C.pp.p, (size_t)(nx + 1) * 8, cudaMemcpyDeviceToHost, s->stream));
    CU(cudaStreamSynchronize(s->stream));
    long long maxrow = 0;
    for (long long q = 0; q < nx; ++q) maxrow = std::max(maxrow, (B.hp[q + 1] - B.hp[q]) * L);
    if (maxrow >= (1LL << 31) - 1)
        return fail(WLSQM_E_VALUE, "one query has %lld candidate slots (pairs x (max nk + 1)); at most 2^31 - 2 are supported", maxrow);
    const int cap_env = env_int("WLSQM_CONT_ROW_CAP", 2048);
    int row_cap = 0;
    if (cap_env > 0) {
        row_cap = 32;
        while (row_cap < cap_env && row_cap < maxrow) row_cap <<= 1;
    }
    B.chunk_slots = std::max<long long>(std::max(env_int("WLSQM_CONT_CHUNK_SLOTS", 1 << 26), 1), maxrow);
    int rc = B.cnt.reserve((size_t)(nx + 1) * 8);
    if (!rc) rc = B.rp.reserve((size_t)(nx + 1) * 8);
    if (rc) return rc;
    P.meta = r->dmeta; P.uni = r->uni; P.nx = nx; P.npairs = C.npairs; P.pair_ptr = (const long long*)C.pp.p; P.J = Jd;
    P.pair_query = (const int*)C.pq.p; P.hoods = (const int32_t*)r->hoods_dev.p; P.hoods_s0 = r->maxnk; P.center = center;
    P.L = (int)L; P.maxnk = r->maxnk; P.row_cap = row_cap; P.cnt = (long long*)B.cnt.p; P.rp = (const long long*)B.rp.p;
    CU(cudaMemsetAsync(B.cnt.p, 0, (size_t)(nx + 1) * 8, s->stream));
    CU(launch_cont_rows(P, false, 32, s->stream));
    if (maxrow > row_cap) {
        // scratch for the largest chunk
        long long slots = 0, nseg = 0;
        cont_chunks(P, B, [&](long long q0, long long q1) {
            slots = std::max(slots, (B.hp[q1] - B.hp[q0]) * L);
            nseg = std::max(nseg, q1 - q0);
            return WLSQM_OK;
        });
        rc = B.seg.reserve((size_t)(nseg + 1) * 4);
        if (!rc) rc = B.keys.reserve((size_t)slots * 4);
        if (!rc) rc = B.keys_s.reserve((size_t)slots * 4);
        if (!rc) rc = B.cand.reserve((size_t)slots * 4);
        if (!rc) rc = B.cand_s.reserve((size_t)slots * 4);
        if (!rc) rc = B.head.reserve((size_t)(slots + 1) * 4);
        if (!rc) rc = B.hpos.reserve((size_t)(slots + 1) * 4);
        if (rc) return rc;
        P.seg = (int*)B.seg.p; P.keys = (unsigned*)B.keys.p; P.cand = (int*)B.cand.p;
        P.keys_sorted = (const unsigned*)B.keys_s.p; P.cand_sorted = (const int*)B.cand_s.p;
        P.head = (int*)B.head.p; P.hpos = (const int*)B.hpos.p;
        P.q0 = 0; P.q1 = nseg; P.nslots = slots;
        size_t tb = 0;
        CU(cont_long_rows(P, false, 32, nullptr, &tb, s->stream));
        rc = B.tmp.reserve(tb + 16);
        if (!rc) rc = cont_chunks(P, B, [&](long long q0, long long q1) { return cont_chunk_run(s, P, B, q0, q1, false, 32); });
        if (rc) return rc;
    }
    size_t tb = 0;
    CU(csr_scan((long long*)B.cnt.p, (long long*)B.rp.p, nx + 1, nullptr, &tb, s->stream));
    DevBuf tmp;
    rc = tmp.reserve(tb + 16);
    if (rc) return rc;
    tb += 16;
    long long total = 0;
    cudaError_t e = csr_scan((long long*)B.cnt.p, (long long*)B.rp.p, nx + 1, tmp.p, &tb, s->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&total, (const long long*)B.rp.p + nx, 8, cudaMemcpyDeviceToHost, s->stream);
    const cudaError_t e2 = cudaStreamSynchronize(s->stream);
    tmp.release();
    if (e == cudaSuccess) e = e2;
    if (e != cudaSuccess) return fail(WLSQM_E_CUDA, "continuous operator pattern: %s", cudaGetErrorString(e));
    P.nnz = total;
    *nnz = total;
    return WLSQM_OK;
}

// fill pass after cont_pattern: rowptr, the short rows, then the chunks of the sort route
static int cont_fill(wlsqm_solver_t* s, ContCsrParams& P, ContPattern& B, int index_bits) {
    CU(launch_cont_rows(P, true, index_bits, s->stream));
    if (!B.tmp.p) return WLSQM_OK;
    return cont_chunks(P, B, [&](long long q0, long long q1) { return cont_chunk_run(s, P, B, q0, q1, true, index_bits); });
}

// rowptr = [0] for nx = 0
static int cont_empty_rowptr(void* rowptr, size_t ib) {
    const long long z = 0;
    if (is_device_ptr(rowptr)) CU(cudaMemcpy(rowptr, &z, ib, cudaMemcpyHostToDevice));
    else memcpy(rowptr, &z, ib);
    return WLSQM_OK;
}

int wlsqm_solver_interp_continuous_count(wlsqm_solver_t* s, const double* x, int64_t x_s0, int64_t nx, double r,
                                         int64_t center, int64_t* pair_ptr, int64_t* npairs, int64_t* nnz) {
    if (!npairs) return fail(WLSQM_E_VALUE, "npairs must not be NULL");
    *npairs = 0;
    if (nnz) *nnz = 0;
    int rc = cont_check(s, nx, r);
    if (rc) return rc;
    if (nnz) {
        const wlsqm_solver* rt = s->lender ? s->lender : s;
        if (!rt->hoods_current)
            return fail(WLSQM_E_NOTREADY, "the global operator needs the neighbour lists of prepare_hoods() as the last prepare");
        rc = opx_center(s, center);
        if (rc) return rc;
    }
    if (nx == 0) return pair_ptr ? cont_empty_rowptr(pair_ptr, 8) : WLSQM_OK;
    rc = use_device(s);
    if (rc) return rc;
    const double* xd;
    long long xs;
    rc = opx_points(s, x, x_s0, nx, &xd, &xs);
    if (rc) return rc;
    ContPairs C;
    ContPattern B;
    DevBuf Jd;
    struct Release {
        wlsqm_solver_t* s; DevBuf* b[12];
        ~Release() { cudaStreamSynchronize(s->stream); for (DevBuf* d : b) d->release(); }
    } release{s, {&C.pp, &C.j32, &C.pq, &C.alpha, &B.seg, &B.keys, &B.cand, &B.keys_s, &B.cand_s, &B.head, &B.hpos, &Jd}};
    struct ReleaseMore {
        wlsqm_solver_t* s; DevBuf* b[3];
        ~ReleaseMore() { cudaStreamSynchronize(s->stream); for (DevBuf* d : b) d->release(); }
    } release_more{s, {&B.cnt, &B.rp, &B.tmp}};
    rc = cont_count(s, xd, xs, nx, r, C);
    if (rc) return rc;
    long long total = 0;
    if (nnz) {
        rc = Jd.reserve((size_t)std::max(C.npairs, 1LL) * 8);
        if (!rc) rc = cont_models(s, xd, xs, nx, r, C, (long long*)Jd.p);
        ContCsrParams P{};
        if (!rc) rc = cont_pattern(s, C, nx, center, (const long long*)Jd.p, B, P, &total);
        if (rc) return rc;
    }
    if (pair_ptr) CU(cudaMemcpyAsync(pair_ptr, C.pp.p, (size_t)(nx + 1) * 8, cudaMemcpyDefault, s->stream));
    CU(cudaStreamSynchronize(s->stream));
    *npairs = C.npairs;
    if (nnz) *nnz = total;
    return WLSQM_OK;
}

// the pairs of x and r after the caller's pair_ptr has been checked, W / K / kf of the pairs, and J in Jd
static int cont_rows(wlsqm_solver_t* s, const double* xd, long long xs, long long nx, double r, const int64_t* pair_ptr,
                     int nops, const double* coeffs, ContPairs& C, DevBuf& sj, int64_t* J, void** Jd, double* W, double* K,
                     double* kf) {
    int rc = cont_same_ptr(s, pair_ptr, C, nx);
    if (rc) return rc;
    rc = opx_out(J, (size_t)C.npairs * 8, sj, Jd);
    if (!rc && !*Jd) {
        rc = sj.reserve((size_t)std::max(C.npairs, 1LL) * 8);
        *Jd = sj.p;
    }
    if (!rc) rc = cont_models(s, xd, xs, nx, r, C, (long long*)*Jd);
    if (!rc && C.npairs)
        rc = opx_interp(s, xd, xs, (const long long*)*Jd, C.npairs, nops, coeffs, W, K, kf, (const int*)C.pq.p,
                        (const double*)C.alpha.p);
    return rc;
}

int wlsqm_solver_interp_continuous_stencils(wlsqm_solver_t* s, const double* x, int64_t x_s0, int64_t nx, double r, int nops,
                                            const double* coeffs, const int64_t* pair_ptr, int64_t* J, double* W, double* K) {
    int rc = opx_check(s, nops, coeffs, false);
    if (!rc) rc = cont_check(s, nx, r);
    if (rc) return rc;
    if (!pair_ptr) return fail(WLSQM_E_VALUE, "pair_ptr must not be NULL");
    if (nx == 0) return WLSQM_OK;
    const double* xd;
    long long xs;
    rc = opx_points(s, x, x_s0, nx, &xd, &xs);
    if (rc) return rc;
    ContPairs C;
    DevBuf sj, sw, sk;
    struct Release {
        wlsqm_solver_t* s; DevBuf* b[7];
        ~Release() { cudaStreamSynchronize(s->stream); for (DevBuf* d : b) d->release(); }
    } release{s, {&C.pp, &C.j32, &C.pq, &C.alpha, &sj, &sw, &sk}};
    rc = cont_count(s, xd, xs, nx, r, C);
    if (rc) return rc;
    const long long np = C.npairs;
    if (np > 0 && !W) return fail(WLSQM_E_VALUE, "W must not be NULL");
    const size_t wb = (size_t)nops * np * s->maxnk * 8, kb = (size_t)nops * np * s->maxno * 8;
    void *Jd, *Wd, *Kd;
    rc = opx_out(np ? W : nullptr, wb, sw, &Wd);
    if (!rc) rc = opx_out(np ? K : nullptr, kb, sk, &Kd);
    if (!rc) rc = cont_rows(s, xd, xs, nx, r, pair_ptr, nops, coeffs, C, sj, J, &Jd, (double*)Wd, (double*)Kd, nullptr);
    if (!rc && np) rc = opx_copy_out(W, Wd, wb, s->stream);
    if (!rc && np && K) rc = opx_copy_out(K, Kd, kb, s->stream);
    if (!rc && np && J) rc = opx_copy_out(J, Jd, (size_t)np * 8, s->stream);
    if (rc) return rc;
    CU(cudaStreamSynchronize(s->stream));
    return WLSQM_OK;
}

int wlsqm_solver_interp_continuous_operator_csr(wlsqm_solver_t* s, const double* x, int64_t x_s0, int64_t nx, double r,
                                                int nops, const double* coeffs, int64_t center, int index_bits,
                                                const int64_t* pair_ptr, int64_t* J, void* rowptr, void* col, double* values,
                                                double* K) {
    int rc = opx_check(s, nops, coeffs, true);
    if (!rc) rc = opx_center(s, center);
    if (!rc) rc = cont_check(s, nx, r);
    if (rc) return rc;
    if (index_bits != 32 && index_bits != 64) return fail(WLSQM_E_VALUE, "index_bits must be 32 or 64, got %d", index_bits);
    if (!rowptr) return fail(WLSQM_E_VALUE, "rowptr must not be NULL");
    if (!pair_ptr) return fail(WLSQM_E_VALUE, "pair_ptr must not be NULL");
    const size_t ib = index_bits / 8;
    if (nx == 0) return cont_empty_rowptr(rowptr, ib);
    const double* xd;
    long long xs;
    rc = opx_points(s, x, x_s0, nx, &xd, &xs);
    if (rc) return rc;
    ContPairs C;
    ContPattern B;
    DevBuf sj, wtmp, kf, s_rp, s_col, s_val, s_k;
    struct Release {
        wlsqm_solver_t* s; DevBuf* b[18];
        ~Release() { cudaStreamSynchronize(s->stream); for (DevBuf* d : b) d->release(); }
    } release{s, {&C.pp, &C.j32, &C.pq, &C.alpha, &B.seg, &B.keys, &B.cand, &B.keys_s, &B.cand_s, &B.head, &B.hpos, &sj,
                  &wtmp, &kf, &s_rp, &s_col, &s_val, &s_k}};
    struct ReleaseMore {
        wlsqm_solver_t* s; DevBuf* b[3];
        ~ReleaseMore() { cudaStreamSynchronize(s->stream); for (DevBuf* d : b) d->release(); }
    } release_more{s, {&B.cnt, &B.rp, &B.tmp}};
    rc = cont_count(s, xd, xs, nx, r, C);
    if (rc) return rc;
    const long long np = C.npairs;
    rc = wtmp.reserve((size_t)nops * std::max(np, 1LL) * std::max(s->maxnk, 1) * 8);
    if (!rc && center >= 0) rc = kf.reserve((size_t)nops * std::max(np, 1LL) * 8);
    if (rc) return rc;
    const size_t kb = (size_t)nops * np * s->maxno * 8;
    void *Jd, *kd;
    rc = opx_out(np ? K : nullptr, kb, s_k, &kd);
    if (!rc) rc = cont_rows(s, xd, xs, nx, r, pair_ptr, nops, coeffs, C, sj, J, &Jd, (double*)wtmp.p, (double*)kd,
                            center >= 0 ? (double*)kf.p : nullptr);
    if (rc) return rc;
    ContCsrParams P{};
    long long nnz = 0;
    rc = cont_pattern(s, C, nx, center, (const long long*)Jd, B, P, &nnz);
    if (rc) return rc;
    if (index_bits == 32 && nnz >= (1LL << 31))
        return fail(WLSQM_E_VALUE, "nnz = %lld does not fit 32-bit indices; use index_bits = 64", nnz);
    if (nnz > 0 && (!col || !values)) return fail(WLSQM_E_VALUE, "col and values must not be NULL");
    const size_t rb = (size_t)(nx + 1) * ib, cb = (size_t)nnz * ib, vb = (size_t)nops * nnz * 8;
    void *rpd, *cd, *vd;
    rc = opx_out(rowptr, rb, s_rp, &rpd);
    if (!rc) rc = opx_out(nnz ? col : nullptr, cb, s_col, &cd);
    if (!rc) rc = opx_out(nnz ? values : nullptr, vb, s_val, &vd);
    if (rc) return rc;
    P.W = (const double*)wtmp.p; P.kf = (const double*)kf.p; P.nops = nops;
    P.rowptr = rpd; P.col = cd; P.values = (double*)vd;
    rc = cont_fill(s, P, B, index_bits);
    if (rc) return rc;
    rc = opx_copy_out(rowptr, rpd, rb, s->stream);
    if (!rc && nnz) rc = opx_copy_out(col, cd, cb, s->stream);
    if (!rc && nnz) rc = opx_copy_out(values, vd, vb, s->stream);
    if (!rc && np && K) rc = opx_copy_out(K, kd, kb, s->stream);
    if (!rc && np && J) rc = opx_copy_out(J, Jd, (size_t)np * 8, s->stream);
    if (rc) return rc;
    CU(cudaStreamSynchronize(s->stream));
    return WLSQM_OK;
}

// Several caller-held solutions at once (wlsqm_interp_fields.cu): wlsqm_solver_interpolate (I given) or
// wlsqm_solver_interpolate_continuous (I == NULL, continuous) per field j of fi [nf][ncases][>= max no].
static int interp_fields_core(wlsqm_solver_t* s, int64_t nf, const double* fi, int64_t fi_sf, int64_t fi_s0, const double* x,
                              int64_t x_s0, const int64_t* I, int64_t nx, bool continuous, double r, int diff, double* out,
                              int64_t out_sf, int64_t out_sq) {
    if (!s) return fail(WLSQM_E_VALUE, "NULL solver");
    if (!s->ready) return fail(WLSQM_E_NOTREADY, "Solver is not in the ready state; prepare() must be called first");
    if (continuous && !s->models_grid)
        return fail(WLSQM_E_NOTREADY, "Points xi have not been indexed; prep_interpolate() must be called before interpolate()");
    if (nf < 0 || nx < 0) return fail(WLSQM_E_VALUE, "nf and nx must be >= 0");
    if (nf == 0 || nx == 0) return WLSQM_OK;
    if (!fi || !x || (!continuous && !I) || !out) return fail(WLSQM_E_VALUE, "fi, x, I and out must not be NULL");
    if (continuous && !(r > 0.0)) return fail(WLSQM_E_VALUE, "r must be positive");
    const int size = number_of_dofs(s->dim, 4);
    const bool all = !continuous && diff == WLSQM_DIFF_ALL;
    if (!all && (diff < 0 || diff >= size)) return fail(WLSQM_E_VALUE, "invalid diff %d", diff);
    const long long n = s->ncases, dim = s->dim, maxno = s->maxno, width = all ? maxno : 1;
    if (n == 0) return fail(WLSQM_E_NOTREADY, "the solver has no models to evaluate");
    if (fi_sf < 0 || fi_s0 < 0 || x_s0 < 0) return fail(WLSQM_E_VALUE, "fi and x strides must be >= 0");
    if (!fields_layout_ok(nf, nx, width, out_sf, out_sq))
        return fail(WLSQM_E_VALUE, "out layout (field stride %lld, query stride %lld) maps two (field, query, slot) entries to "
                    "one element; use fields-outer (out_sf >= (nx-1)*out_sq + width, out_sq >= width) or fields-inner "
                    "(out_sf >= width, out_sq >= (nf-1)*out_sf + width) rows, width %lld", (long long)out_sf,
                    (long long)out_sq, width);
    int rc = use_device(s);
    if (rc) return rc;
    cudaStream_t st = s->stream;
    const bool fi_dev = is_device_ptr(fi), x_dev = is_device_ptr(x), I_dev = !continuous && is_device_ptr(I);
    const bool out_dev = is_device_ptr(out);
    // elements spanned by each strided array (all strides are non-negative)
    const long long fi_span = (nf - 1) * fi_sf + (n - 1) * fi_s0 + maxno;
    const long long out_span = (nf - 1) * out_sf + (nx - 1) * out_sq + width;
    if (out_dev) {
        if ((fi_dev && ranges_overlap(out, out_span * 8, fi, fi_span * 8)) ||
            (x_dev && ranges_overlap(out, out_span * 8, x, ((nx - 1) * x_s0 + dim) * 8)) ||
            (I_dev && ranges_overlap(out, out_span * 8, I, nx * 8)))
            return fail(WLSQM_E_VALUE, "device out overlaps device fi, x or I");
    }

    InterpFieldsParams F{};
    InterpParams& P = F.P;
    P.dim = s->dim; P.nx = nx; P.diff = all ? -1 : diff; P.nmodels = n;
    P.xi = s->xi_dev; P.xi_s0 = s->dim;
    P.order = s->dorder; P.order_uniform = s->uni.order;
    F.width = (int)width;
    // fi rows that are not dense (fields-inner, pitched) are copied to dense rows, one pass at a time right before the
    // pass: the rows of one field then share L2 lines with no other field's, and the rows just written are still largely
    // in L2 when the pass reads them.  Read in place, fields-inner rows at 1M models and 16M queries took 2.7 to 3.4 times
    // the time of dense ones (profiles/r08_interp_fields_plans.txt).  Host fi is staged the same way, per pass; host rows
    // that overlap (fi_s0 < max no) are staged whole as one span, strides kept.
    const double* fi_use = fi;
    const bool compact = fi_s0 >= maxno && (!fi_dev || (fi_s0 != maxno && n > 1));
    if (!compact && !fi_dev) {
        rc = s->st_fi.reserve((size_t)fi_span * 8);
        if (rc) return rc;
        rc = to_dense((double*)s->st_fi.p, fi, 1, fi_span, fi_span, st);
        if (rc) return rc;
        fi_use = (const double*)s->st_fi.p;
    }
    if (x_dev) { P.x = x; P.x_s0 = x_s0; }
    else {
        rc = s->st_x.reserve((size_t)nx * dim * 8);
        if (rc) return rc;
        rc = stage_in(s->device, (double*)s->st_x.p, x, nx, dim, x_s0, st);
        if (rc) return rc;
        P.x = (const double*)s->st_x.p; P.x_s0 = dim;
    }
    if (!continuous) {
        if (I_dev) P.I = (const long long*)I;
        else {
            rc = s->st_I.reserve((size_t)nx * 8);
            if (rc) return rc;
            rc = stage_in(s->device, (double*)s->st_I.p, reinterpret_cast<const double*>(I), nx, 1, 1, st);   // (8-byte items)
            if (rc) return rc;
            P.I = (const long long*)s->st_I.p;
        }
    }
    double* out_use = out;
    long long out_sf_use = out_sf;
    if (out_dev) P.out_s0 = out_sq;
    else {
        rc = s->st_out.reserve((size_t)nf * nx * width * 8);
        if (rc) return rc;
        out_use = (double*)s->st_out.p; out_sf_use = nx * width; P.out_s0 = width;
    }
    P.stage_no = (all && s->uniform_no && P.out_s0 == s->uni.no) ? s->uni.no : 0;

    // fields per pass from the byte model of wlsqm_interp_fields.cu
    if (!s->l2_bytes) CU(cudaDeviceGetAttribute(&s->l2_bytes, cudaDevAttrL2CacheSize, s->device));
    double rows_per_query = 1.0, query_bytes = 8.0 * dim + 8.0;
    GridView g{};
    if (continuous) {
        // models in a ball of radius r and candidates in its cell box, for a uniform density over the grid's box
        g = grid_view(s->models_grid);
        double box = 1.0, ball = 1.0, cells = 1.0;
        for (int d = 0; d < dim; ++d) { box *= g.dims[d] * g.h; ball *= r; cells *= 2.0 * r + g.h; }
        ball *= dim == 1 ? 2.0 : (dim == 2 ? 3.141592653589793 : 4.0 / 3.0 * 3.141592653589793);
        rows_per_query = std::min((double)n, std::max(1.0, n * ball / box));
        query_bytes = 8.0 * dim + std::min((double)n, n * cells / box) * (8.0 * dim + 4.0);
    }
    const int fb = interp_fields_per_pass(nf, n, s->maxno, nx, rows_per_query, query_bytes, 8.0 * width, s->l2_bytes);
    if (compact) {
        rc = s->st_fi.reserve((size_t)std::min<long long>(fb, nf) * n * maxno * 8);
        if (rc) return rc;
    }
    for (long long p0 = 0; p0 < nf; p0 += fb) {
        F.nf = (int)std::min<long long>(fb, nf - p0);
        if (compact) {
            double* dense = (double*)s->st_fi.p;
            if (fi_dev) CU(launch_compact_rows(fi + p0 * fi_sf, fi_sf, fi_s0, F.nf, n, (int)maxno, dense, st));
            else {
                for (int j = 0; j < F.nf; ++j) {
                    rc = to_dense(dense + j * n * maxno, fi + (p0 + j) * fi_sf, n, maxno, fi_s0, st);
                    if (rc) return rc;
                }
            }
            P.fi = dense; P.fi_s0 = maxno; F.fi_sf = n * maxno;
        } else {
            P.fi = fi_use + p0 * fi_sf; P.fi_s0 = fi_s0; F.fi_sf = fi_sf;
        }
        P.out = out_use + p0 * out_sf_use; F.out_sf = out_sf_use;
        if (F.nf == 1 && !all && P.out_s0 == 1) {
            // one field in this pass, dense one-slot output: the single-field kernel and its launch shape serve it
            CU(continuous ? launch_interpolate_continuous(P, g, r, st) : launch_interpolate(P, st));
        } else {
            CU(continuous ? launch_interpolate_continuous_fields(F, g, r, st) : launch_interpolate_fields(F, st));
        }
    }
    if (!out_dev) {
        for (long long j = 0; j < nf; ++j) {
            rc = stage_out(s->device, out + j * out_sf, out_sq, (const double*)s->st_out.p + j * nx * width, width, nx, width, st);
            if (rc) return rc;
        }
    }
    if (!fi_dev || !x_dev || (!continuous && !I_dev) || !out_dev) CU(cudaStreamSynchronize(st));
    return WLSQM_OK;
}

int wlsqm_solver_interpolate_fields(wlsqm_solver_t* s, int64_t nf, const double* fi, int64_t fi_sf, int64_t fi_s0,
                                    const double* x, int64_t x_s0, const int64_t* I, int64_t nx, int diff, double* out,
                                    int64_t out_sf, int64_t out_sq) {
    return interp_fields_core(s, nf, fi, fi_sf, fi_s0, x, x_s0, I, nx, false, 0.0, diff, out, out_sf, out_sq);
}

int wlsqm_solver_interpolate_continuous_fields(wlsqm_solver_t* s, int64_t nf, const double* fi, int64_t fi_sf,
                                               int64_t fi_s0, const double* x, int64_t x_s0, int64_t nx, double r, int diff,
                                               double* out, int64_t out_sf, int64_t out_sq) {
    return interp_fields_core(s, nf, fi, fi_sf, fi_s0, x, x_s0, nullptr, nx, true, r, diff, out, out_sf, out_sq);
}

// One-shot fits without sensitivities on a uniform batch: one launch of the fused kernel (assemble, equilibrate,
// factor, solve; no operator is formed, nothing is kept).  Returns 1 if the call was handled (rc_out has the result),
// 0 if the batch does not qualify and the general path (create + prepare + solve + destroy) must run.
static int fit_many_direct(int dimension, int64_t ncases, const double* xk, int64_t xk_s0, int64_t xk_s1, const double* fk,
                           int64_t fk_s0, int64_t fk_s1, const int32_t* nk, const double* xi, int64_t xi_s0, double* fi,
                           int64_t fi_s0, const int32_t* order, const int64_t* knowns, const int32_t* wm, int device,
                           int* rc_out) {
    if (env_int("WLSQM_FIT_DIRECT", 1) == 0) return 0;
    if (ncases < 1 || dimension < 1 || dimension > 3 || !nk || !order || !knowns || !wm || !xk || !fk || !xi || !fi) return 0;
    if (!scan_meta(ncases, nk, order, knowns, wm).uniform()) return 0;
    const int no = number_of_dofs(dimension, order[0]);
    if (no < 0 || nk[0] < 0 || (wm[0] != WLSQM_WEIGHT_UNIFORM && wm[0] != WLSQM_WEIGHT_CENTER)) return 0;   // general path reports it
    if (!prepare_reg_direct_ok(dimension, order[0])) return 0;
    if (wlsqm_device_count() < 1 || device < 0 || device >= wlsqm_device_count()) return 0;
    const bool xk_dev = is_device_ptr(xk), fk_dev = is_device_ptr(fk), xi_dev = is_device_ptr(xi), fi_dev = is_device_ptr(fi);
    const int dim = dimension, k = nk[0];
    if (!xk_dev && xk_s1 != dim && k > 1) return 0;
    if (!fk_dev && fk_s1 != 1 && k > 1) return 0;
    if (xk_dev && xk_s1 != dim) return 0;                      // (the kernel wants contiguous neighbour rows)
    if (fk_dev && fi_dev) {
        // fk may be a view of fi (the deferred write-back of expert.pyx:548-557 exists for that): general path
        const char *a0 = (const char*)fk, *a1 = a0 + ((ncases - 1) * fk_s0 + (long long)(k - 1) * fk_s1 + 1) * 8;
        const char *b0 = (const char*)fi, *b1 = b0 + ((ncases - 1) * fi_s0 + no) * 8;
        if (a0 < b1 && b0 < a1) return 0;
    }
    // a solver shell for the launch configuration only (no device state)
    wlsqm_solver sh;
    sh.dim = dim; sh.device = device; sh.ncases = ncases;
    CaseMeta m;
    memset(&m, 0, sizeof m);
    m.knowns = knowns[0] & ((1LL << no) - 1);
    m.nkn = (signed char)__builtin_popcountll((unsigned long long)m.knowns);
    m.nk = k; m.no = (short)no; m.nr = (short)(no - m.nkn); m.order = (signed char)order[0]; m.wm = (signed char)wm[0];
    sh.uni = m;
    sh.maxnk = k; sh.maxno = no; sh.maxnr = m.nr; sh.maxnq = k + m.nkn; sh.maxorder = m.order; sh.maxnkn = m.nkn;
    auto run = [&]() -> int {
        CU(cudaSetDevice(device));
        int smc = 0;
        if (cudaDeviceGetAttribute(&smc, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && smc > 0) sh.sm_count = smc;
        else cudaGetLastError();
        cudaStream_t st = caller_stream();   // the caller's stream (default: the legacy default stream); synchronous result
        DevBuf bxk, bfk, bxi, bfi;
        auto done = [&](int r) { bxk.release(); bfk.release(); bxi.release(); bfi.release(); return r; };
        int rc = WLSQM_OK;
        PrepRegParams R{};
        R.meta = nullptr; R.uni = m; R.op_stride = 0; R.ncases = ncases; R.geom_uniform = 1; R.op = nullptr;
        R.xi = xi; R.xi_s0 = xi_s0; R.xk = xk; R.xk_s0 = xk_s0; R.xk_s1 = xk_s1;
        R.fk = fk; R.fk_s0 = fk_s0; R.fk_s1 = fk_s1; R.fi = fi; R.fi_s0 = fi_s0;
        if (!xk_dev) {
            rc = bxk.reserve((size_t)ncases * k * dim * 8);
            if (!rc) rc = stage_in(device, (double*)bxk.p, xk, ncases, (long long)k * dim, xk_s0, st);
            R.xk = (const double*)bxk.p; R.xk_s0 = (long long)k * dim; R.xk_s1 = dim;
        }
        if (!rc && !fk_dev) {
            rc = bfk.reserve((size_t)ncases * k * 8);
            if (!rc) rc = stage_in(device, (double*)bfk.p, fk, ncases, k, fk_s0, st);
            R.fk = (const double*)bfk.p; R.fk_s0 = k; R.fk_s1 = 1;
        }
        if (!rc && !xi_dev) {
            rc = bxi.reserve((size_t)ncases * dim * 8);
            if (!rc) rc = to_dense((double*)bxi.p, xi, ncases, dim, xi_s0, st);
            R.xi = (const double*)bxi.p; R.xi_s0 = dim;
        }
        if (!rc && !fi_dev) {
            rc = bfi.reserve((size_t)ncases * no * 8);
            if (!rc) rc = stage_in(device, (double*)bfi.p, fi, ncases, no, fi_s0, st);      // the known values travel in
            R.fi = (double*)bfi.p; R.fi_s0 = no;
        }
        if (rc) return done(rc);
        LaunchCfg L;
        if (!config_prepare_reg(&sh, R, L, true)) return done(-1000);          // does not fit: general path
        cudaError_t e = launch_prepare_reg(dim, m.order, R, L.blocks, L.threads, L.smem, st);
        if (e == cudaSuccess && !fi_dev) {
            rc = stage_out(device, fi, fi_s0, (const double*)bfi.p, no, ncases, no, st);
            if (rc) return done(rc);
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) return done(fail(WLSQM_E_CUDA, "one-shot fit: %s", cudaGetErrorString(e)));
        return done(WLSQM_OK);
    };
    const int rc = run();
    if (rc == -1000) return 0;
    *rc_out = rc;
    return 1;
}

int wlsqm_fit_many(int dimension, int64_t ncases, const double* xk, int64_t xk_s0, int64_t xk_s1, const double* fk,
                   int64_t fk_s0, int64_t fk_s1, const int32_t* nk, const double* xi, int64_t xi_s0, double* fi,
                   int64_t fi_s0, double* sens, int64_t sens_s0, int64_t sens_s1, int do_sens, const int32_t* order,
                   const int64_t* knowns, const int32_t* wm, int algorithm, int max_iter, int device,
                   int32_t* iters_out) {
    if (algorithm == WLSQM_ALGO_BASIC && !do_sens) {
        int rc = WLSQM_OK;
        if (fit_many_direct(dimension, ncases, xk, xk_s0, xk_s1, fk, fk_s0, fk_s1, nk, xi, xi_s0, fi, fi_s0, order, knowns,
                            wm, device, &rc)) {
            if (iters_out) *iters_out = 0;
            return rc;
        }
    }
    wlsqm_solver_t* s = nullptr;
    int rc = wlsqm_solver_create(dimension, ncases, nk, order, knowns, wm, algorithm, do_sens, max_iter, 0, device, &s);
    if (rc) return rc;
    // the temporary solver works on its own stream: order it after what the caller has queued (device-array arguments
    // may still be being produced, or their blocks still be in use, on the caller's stream)
    if (order_after_caller(s->stream) != cudaSuccess) { cudaGetLastError(); cudaStreamSynchronize(caller_stream()); }
    rc = wlsqm_solver_prepare(s, xi, xi_s0, xk, xk_s0, xk_s1);
    if (!rc) rc = wlsqm_solver_solve(s, fk, fk_s0, fk_s1, fi, fi_s0, sens, sens_s0, sens_s1, iters_out);
    if (!rc) rc = wlsqm_solver_synchronize(s);
    std::string keep = g_err;
    wlsqm_solver_destroy(s);
    g_err = keep;
    return rc;
}

int wlsqm_interpolate_fit(int dimension, int order, const double* xi, const double* fi, const double* x, int64_t x_s0,
                          int64_t nx, int diff, double* out, int device) {
    if (dimension < 1 || dimension > 3) return fail(WLSQM_E_VALUE, "dimension must be 1, 2 or 3; got %d", dimension);
    const int no = number_of_dofs(dimension, order);
    if (no < 0) return fail(WLSQM_E_VALUE, "order must be 0, 1, 2, 3 or 4; got %d", order);
    const int size = number_of_dofs(dimension, 4);
    if (diff != WLSQM_DIFF_ALL && (diff < 0 || diff >= size)) return fail(WLSQM_E_VALUE, "invalid diff %d", diff);
    if (nx == 0) return WLSQM_OK;
    if (!xi || !fi || !x || !out) return fail(WLSQM_E_VALUE, "NULL argument");
    if (wlsqm_device_count() < 1) return fail(WLSQM_E_CUDA, "no CUDA device available (there is no CPU fallback)");
    CU(cudaSetDevice(device));
    const long long ow = diff == WLSQM_DIFF_ALL ? no : 1;
    DevBuf bm, bx, bo;
    int rc = bm.reserve((size_t)(dimension + no) * 8);
    if (!rc && !is_device_ptr(x)) rc = bx.reserve((size_t)nx * dimension * 8);
    if (!rc && !is_device_ptr(out)) rc = bo.reserve((size_t)nx * ow * 8);
    auto done = [&](int r) { bm.release(); bx.release(); bo.release(); return r; };
    if (rc) return done(rc);
    cudaStream_t st = caller_stream();
    double* dm = (double*)bm.p;
    cudaError_t e = cudaMemcpyAsync(dm, xi, (size_t)dimension * 8, cudaMemcpyDefault, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dm + dimension, fi, (size_t)no * 8, cudaMemcpyDefault, st);
    if (e != cudaSuccess) return done(fail(WLSQM_E_CUDA, "interpolate_fit upload: %s", cudaGetErrorString(e)));
    InterpParams P{};
    P.dim = dimension; P.nx = nx; P.diff = diff; P.I = nullptr;
    P.xi = dm; P.xi_s0 = dimension; P.fi = dm + dimension; P.fi_s0 = no; P.order = nullptr; P.order_uniform = order;
    if (bx.p) {
        rc = to_dense((double*)bx.p, x, nx, dimension, x_s0, st);
        if (rc) return done(rc);
        P.x = (const double*)bx.p; P.x_s0 = dimension;
    } else { P.x = x; P.x_s0 = x_s0; }
    P.out = bo.p ? (double*)bo.p : out; P.out_s0 = ow;
    P.stage_no = diff == WLSQM_DIFF_ALL ? no : 0;
    e = launch_interpolate(P, st);
    if (e == cudaSuccess && bo.p) e = cudaMemcpyAsync(out, bo.p, (size_t)nx * ow * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return done(fail(WLSQM_E_CUDA, "interpolate_fit: %s", cudaGetErrorString(e)));
    return done(WLSQM_OK);
}

static int lapack_common(int n, int64_t nlhs, double* A, int32_t* ipiv, double* b, int device, int do_factor, int do_solve,
                         int sym = 0) {
    if (n < 0 || nlhs < 0) return fail(WLSQM_E_VALUE, "n and nlhs must be >= 0");
    if (n == 0 || nlhs == 0) return WLSQM_OK;
    if (wlsqm_device_count() < 1) return fail(WLSQM_E_CUDA, "no CUDA device available (there is no CPU fallback)");
    CU(cudaSetDevice(device));
    const size_t na = (size_t)n * n * nlhs * 8, np = (size_t)n * nlhs * 4, nb = (size_t)n * nlhs * 8;
    DevBuf ba, bp, bb;
    // ipiv may be NULL for the symmetric dsysv driver (the reference's msymmetric keeps its pivots to itself)
    const bool a_dev = is_device_ptr(A), p_dev = ipiv ? is_device_ptr(ipiv) != 0 : true, b_dev = b ? is_device_ptr(b) != 0 : true;
    int rc = WLSQM_OK;
    if (!a_dev) rc = ba.reserve(na);
    if (!rc && !p_dev) rc = bp.reserve(np);
    if (!rc && !b_dev) rc = bb.reserve(nb);
    auto done = [&](int r) { ba.release(); bp.release(); bb.release(); return r; };
    if (rc) return done(rc);
    cudaStream_t st = caller_stream();
    double* dA = a_dev ? A : (double*)ba.p;
    int* dP = p_dev ? ipiv : (int*)bp.p;
    double* dB = b_dev ? b : (double*)bb.p;
    cudaError_t e = cudaSuccess;
    if (!a_dev) e = cudaMemcpyAsync(dA, A, na, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && !p_dev && !do_factor) e = cudaMemcpyAsync(dP, ipiv, np, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && do_solve && !b_dev) e = cudaMemcpyAsync(dB, b, nb, cudaMemcpyHostToDevice, st);
    if (sym) {
        if (e == cudaSuccess) e = launch_sy(n, nlhs, dA, dP, do_solve ? dB : nullptr, do_factor, st);
    } else {
        if (e == cudaSuccess && do_factor && do_solve) e = launch_gesv(n, nlhs, dA, dP, dB, st);
        else if (e == cudaSuccess && do_factor) e = launch_getrf(n, nlhs, dA, dP, st);
        else if (e == cudaSuccess && do_solve) e = launch_getrs(n, nlhs, dA, dP, dB, st);
    }
    if (e == cudaSuccess && do_factor && !a_dev) e = cudaMemcpyAsync(A, dA, na, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && do_factor && !p_dev && ipiv) e = cudaMemcpyAsync(ipiv, dP, np, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && do_solve && !b_dev) e = cudaMemcpyAsync(b, dB, nb, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e == cudaErrorInvalidValue) return done(fail(WLSQM_E_VALUE, "n = %d is too large for the shared-memory LU", n));
    if (e != cudaSuccess) return done(fail(WLSQM_E_CUDA, "batched LU: %s", cudaGetErrorString(e)));
    return done(WLSQM_OK);
}

int wlsqm_mgetrf(int n, int64_t nlhs, double* A, int32_t* ipiv, int device) {
    if (!A || !ipiv) return fail(WLSQM_E_VALUE, "NULL argument");
    return lapack_common(n, nlhs, A, ipiv, nullptr, device, 1, 0);
}
int wlsqm_mgetrs(int n, int64_t nlhs, const double* LU, const int32_t* ipiv, double* b, int device) {
    if (!LU || !ipiv || !b) return fail(WLSQM_E_VALUE, "NULL argument");
    return lapack_common(n, nlhs, const_cast<double*>(LU), const_cast<int32_t*>(ipiv), b, device, 0, 1);
}
int wlsqm_mgesv(int n, int64_t nlhs, double* A, int32_t* ipiv, double* b, int device) {
    if (!A || !ipiv || !b) return fail(WLSQM_E_VALUE, "NULL argument");
    return lapack_common(n, nlhs, A, ipiv, b, device, 1, 1);
}

int wlsqm_msytrf(int n, int64_t nlhs, double* A, int32_t* ipiv, int device) {
    if (!A || !ipiv) return fail(WLSQM_E_VALUE, "NULL argument");
    return lapack_common(n, nlhs, A, ipiv, nullptr, device, 1, 0, 1);
}
int wlsqm_msytrs(int n, int64_t nlhs, const double* UDU, const int32_t* ipiv, double* b, int device) {
    if (!UDU || !ipiv || !b) return fail(WLSQM_E_VALUE, "NULL argument");
    return lapack_common(n, nlhs, const_cast<double*>(UDU), const_cast<int32_t*>(ipiv), b, device, 0, 1, 1);
}
int wlsqm_msysv(int n, int64_t nlhs, double* A, int32_t* ipiv, double* b, int device) {
    if (!A || !b) return fail(WLSQM_E_VALUE, "NULL argument");
    return lapack_common(n, nlhs, A, ipiv, b, device, 1, 1, 1);
}
// tridiag (lapackdrivers.pyx:854-877): DGTSV with one right-hand side; a = DL (n-1 used), b = D (n), c = DU (n-1 used), x = RHS
int wlsqm_gtsv(int n, double* dl, double* d, double* du, double* b, int device) {
    if (n < 0) return fail(WLSQM_E_VALUE, "n must be >= 0");
    if (n == 0) return WLSQM_OK;
    if (!dl || !d || !du || !b) return fail(WLSQM_E_VALUE, "NULL argument");
    if (wlsqm_device_count() < 1) return fail(WLSQM_E_CUDA, "no CUDA device available (there is no CPU fallback)");
    CU(cudaSetDevice(device));
    const bool dev = is_device_ptr(dl) && is_device_ptr(d) && is_device_ptr(du) && is_device_ptr(b);
    const bool host = !is_device_ptr(dl) && !is_device_ptr(d) && !is_device_ptr(du) && !is_device_ptr(b);
    if (!dev && !host) return fail(WLSQM_E_VALUE, "tridiag: the four arrays must live on the same side (host or device)");
    cudaStream_t st = caller_stream();
    const size_t nb = (size_t)n * 8;
    DevBuf buf;
    double *p0 = dl, *p1 = d, *p2 = du, *p3 = b;
    if (host) {
        int rc = buf.reserve(4 * nb);
        if (rc) return rc;
        p0 = (double*)buf.p; p1 = p0 + n; p2 = p1 + n; p3 = p2 + n;
        cudaError_t e = cudaMemcpyAsync(p0, dl, nb, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(p1, d, nb, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(p2, du, nb, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(p3, b, nb, cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) { buf.release(); return fail(WLSQM_E_CUDA, "tridiag upload: %s", cudaGetErrorString(e)); }
    }
    cudaError_t e = launch_gtsv(n, p0, p1, p2, p3, st);
    if (e == cudaSuccess && host) {
        e = cudaMemcpyAsync(dl, p0, nb, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d, p1, nb, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(du, p2, nb, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(b, p3, nb, cudaMemcpyDeviceToHost, st);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    buf.release();
    if (e != cudaSuccess) return fail(WLSQM_E_CUDA, "tridiag: %s", cudaGetErrorString(e));
    return WLSQM_OK;
}

// do_rescale (lapackdrivers.pyx:319-385) over a batch: scale every matrix in place, return the scale vectors
int wlsqm_mrescale(int nrows, int ncols, int64_t nlhs, double* A, int algo, double* row_scale, double* col_scale, int32_t* ok,
                   int device) {
    if (nrows < 0 || ncols < 0 || nlhs < 0) return fail(WLSQM_E_VALUE, "nrows, ncols and nlhs must be >= 0");
    if (algo < 1 || algo > 6) return fail(WLSQM_E_VALUE, "Unknown algorithm identifier, got %d", algo);
    if (nrows == 0 || ncols == 0 || nlhs == 0) return WLSQM_OK;
    if (!A || !row_scale || !col_scale) return fail(WLSQM_E_VALUE, "NULL argument");
    if (wlsqm_device_count() < 1) return fail(WLSQM_E_CUDA, "no CUDA device available (there is no CPU fallback)");
    CU(cudaSetDevice(device));
    const size_t na = (size_t)nrows * ncols * nlhs * 8, nr = (size_t)nrows * nlhs * 8, nc = (size_t)ncols * nlhs * 8, nk = (size_t)nlhs * 4;
    const bool a_dev = is_device_ptr(A), r_dev = is_device_ptr(row_scale), c_dev = is_device_ptr(col_scale);
    const bool k_dev = ok ? is_device_ptr(ok) != 0 : true;
    DevBuf ba, br, bc, bk;
    int rc = WLSQM_OK;
    if (!a_dev) rc = ba.reserve(na);
    if (!rc && !r_dev) rc = br.reserve(nr);
    if (!rc && !c_dev) rc = bc.reserve(nc);
    if (!rc && !k_dev) rc = bk.reserve(nk);
    auto done = [&](int r) { ba.release(); br.release(); bc.release(); bk.release(); return r; };
    if (rc) return done(rc);
    cudaStream_t st = caller_stream();
    double* dA = a_dev ? A : (double*)ba.p;
    double* dR = r_dev ? row_scale : (double*)br.p;
    double* dC = c_dev ? col_scale : (double*)bc.p;
    int* dK = ok ? (k_dev ? ok : (int*)bk.p) : nullptr;
    cudaError_t e = cudaSuccess;
    if (!a_dev) e = cudaMemcpyAsync(dA, A, na, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = launch_rescale(nrows, ncols, nlhs, dA, algo, dR, dC, dK, st);
    if (e == cudaSuccess && !a_dev) e = cudaMemcpyAsync(A, dA, na, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && !r_dev) e = cudaMemcpyAsync(row_scale, dR, nr, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && !c_dev) e = cudaMemcpyAsync(col_scale, dC, nc, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && ok && !k_dev) e = cudaMemcpyAsync(ok, dK, nk, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e == cudaErrorInvalidValue) return done(fail(WLSQM_E_VALUE, "a %d x %d matrix is too large for the shared-memory scaler", nrows, ncols));
    if (e != cudaSuccess) return done(fail(WLSQM_E_CUDA, "batched rescale: %s", cudaGetErrorString(e)));
    return done(WLSQM_OK);
}

int wlsqm_msymmetrize(int n, int64_t nlhs, double* A, int device) {
    if (n < 0 || nlhs < 0) return fail(WLSQM_E_VALUE, "n and nlhs must be >= 0");
    if (n == 0 || nlhs == 0) return WLSQM_OK;
    if (!A) return fail(WLSQM_E_VALUE, "NULL argument");
    if (wlsqm_device_count() < 1) return fail(WLSQM_E_CUDA, "no CUDA device available (there is no CPU fallback)");
    CU(cudaSetDevice(device));
    const size_t na = (size_t)n * n * nlhs * 8;
    const bool a_dev = is_device_ptr(A);
    DevBuf ba;
    if (!a_dev) { int rc = ba.reserve(na); if (rc) return rc; }
    cudaStream_t st = caller_stream();
    double* dA = a_dev ? A : (double*)ba.p;
    cudaError_t e = cudaSuccess;
    if (!a_dev) e = cudaMemcpyAsync(dA, A, na, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = launch_symmetrize(n, nlhs, dA, st);
    if (e == cudaSuccess && !a_dev) e = cudaMemcpyAsync(A, dA, na, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    ba.release();
    if (e != cudaSuccess) return fail(WLSQM_E_CUDA, "msymmetrize: %s", cudaGetErrorString(e));
    return WLSQM_OK;
}

}  // extern "C"
