/*
 * wlsqm_b200.h -- C ABI of the B200-native wlsqm hot path (libwlsqm_b200.so).
 *
 * This is the drop-in boundary: plain pointers, sizes and strides, no torch / numpy types.
 * Every entry point names the reference interface it replaces (paths relative to the root of
 * Technologicat/python-wlsqm).  The reference has no FFI of its own -- its boundary is the Python
 * surface of four Cython modules (wlsqm/__init__.py:25-28) -- so these functions are what a thin
 * Cython / ctypes shim behind those Python names binds (INTEGRATION.md shows that shim).
 *
 * Conventions
 *   - All data is float64; nk/order/weighting_method are int32, knowns int64 (simple.pyx:149-159).
 *   - Strides are in ELEMENTS, not bytes.  The last axis of xi/xk/fi/sens is contiguous, exactly as
 *     the reference's memoryview signatures demand; fk may be strided on both axes.
 *   - Data pointers (xi, xk, fk, fi, sens, x, I, out, A, b, ipiv) may be HOST or DEVICE memory; the
 *     library asks the CUDA runtime which.  Device pointers are used in place (zero copy, work is
 *     enqueued on the solver's stream and the call returns without synchronising unless it has to
 *     return a value).  Host pointers are staged through device buffers owned by the library and
 *     the call returns when the results are in host memory.  Host arrays must have a unit stride on
 *     their last axis (fk included) -- rows may be pitched.
 *   - Metadata pointers (nk, order, knowns, weighting_method) are always HOST memory.
 *   - Return value: 0 on success, otherwise one of WLSQM_E_*; wlsqm_last_error() has the message.
 *     The Python shim maps WLSQM_E_VALUE -> ValueError, WLSQM_E_MEMORY -> MemoryError,
 *     WLSQM_E_NOTREADY / WLSQM_E_CUDA -> RuntimeError (the reference's exception surface,
 *     expert.pyx:131-189,493-494,673-674,742-743).
 *   - There is no CPU fallback: without a CUDA device every compute entry point fails with WLSQM_E_CUDA.
 */
#ifndef WLSQM_B200_H
#define WLSQM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define WLSQM_API __attribute__((visibility("default")))
#else
#define WLSQM_API
#endif

#define WLSQM_OK 0
#define WLSQM_E_VALUE (-1)
#define WLSQM_E_MEMORY (-2)
#define WLSQM_E_CUDA (-3)
#define WLSQM_E_NOTREADY (-4)

/* wlsqm/fitter/defs.pyx:69-75 */
#define WLSQM_ALGO_BASIC 1
#define WLSQM_ALGO_ITERATIVE 2
#define WLSQM_WEIGHT_UNIFORM 1
#define WLSQM_WEIGHT_CENTER 2

/* interpolate: evaluate every derivative slot of the model in one pass (extension, out is [nx][out_s0]) */
#define WLSQM_DIFF_ALL (-1)

typedef struct wlsqm_solver wlsqm_solver_t;

/* ---- library ---------------------------------------------------------------------------------- */
WLSQM_API int wlsqm_b200_abi_version(void);
WLSQM_API const char* wlsqm_last_error(void);                 /* thread-local message of the last failure */
WLSQM_API int wlsqm_device_count(void);                       /* CUDA devices visible; 0 if none */

/* number_of_dofs: wlsqm/fitter/infra.pyx:67-112, exported as wlsqm/fitter/expert.pyx:57-63.
 * Returns -1 for a bad dimension, -2 for a bad order (no error state is set). */
WLSQM_API int wlsqm_number_of_dofs(int dimension, int order);

/* max nk, min / max order and "every case alike" of the per-case metadata arrays (host memory), in one pass: what the
 * Python mirror needs for the shape checks of simple.pyx:149-159 / expert.pyx:131-159 without several array reductions */
WLSQM_API int wlsqm_meta_summary(int64_t ncases, const int32_t* nk, const int32_t* order, const int64_t* knowns,
                       const int32_t* weighting_method, int32_t* max_nk, int32_t* min_order, int32_t* max_order,
                       int32_t* uniform);

/* page-locked host buffers for the staged (host-pointer) path */
WLSQM_API void* wlsqm_pinned_alloc(int64_t bytes);
WLSQM_API void* wlsqm_pinned_alloc_wc(int64_t bytes);          /* write-combined: for buffers the host only writes */
WLSQM_API void wlsqm_pinned_free(void* p);

/* Device memory of the library comes from one stream-ordered CUDA memory pool per device: what a destroyed solver or
 * a finished one-shot fit gives back stays cached (up to WLSQM_POOL_KEEP_MB, default 8192; WLSQM_POOL=0 disables the
 * pool) so that the next call does not pay cudaMalloc / cudaFree -- the counterpart of the reference building its
 * per-call arena with one malloc (CaseManager_commit, wlsqm/fitter/infra.pyx:545-632).  stats: bytes reserved from
 * the driver / in use (-1 before the first allocation on that device); trim: return the cached blocks. */
WLSQM_API int wlsqm_pool_stats(int device, int64_t* reserved, int64_t* used);
WLSQM_API int wlsqm_pool_trim(int device);

/* ---- ExpertSolver: wlsqm/fitter/expert.pyx:66-781 ------------------------------------------------ */

/* ExpertSolver.__init__ (expert.pyx:92-263) + CaseManager_new/Case_new/commit (infra.pyx:308-471,545-632).
 * `device` is the CUDA ordinal that will own the solver's state.  ntasks has no meaning here. */
WLSQM_API int wlsqm_solver_create(int dimension, int64_t ncases, const int32_t* nk, const int32_t* order,
                        const int64_t* knowns, const int32_t* weighting_method, int algorithm, int do_sens,
                        int max_iter, int debug, int device, wlsqm_solver_t** out);

/* ExpertSolver(..., host=other): guest mode (expert.pyx:163-189,243-263; Case_new(host=...) infra.pyx:528-544).  The
 * guest borrows the host's prepared state (operators, per-case records, origins) and owns only its solution copy:
 * several fields on one geometry cost one set of operators.  Sizes and debug flag are the host's; algorithm, do_sens,
 * max_iter are the guest's own (an ALGO_ITERATIVE guest needs an ALGO_ITERATIVE host).  The host must outlive the guest.
 * wlsqm_solver_prepare on a guest (or wlsqm_solver_prepare_guest) computes nothing and marks it ready. */
WLSQM_API int wlsqm_solver_create_guest(wlsqm_solver_t* host, int algorithm, int do_sens, int max_iter, wlsqm_solver_t** out);
WLSQM_API int wlsqm_solver_prepare_guest(wlsqm_solver_t* s);

/* ExpertSolver.__del__ (expert.pyx:267-286) / CaseManager_del (infra.pyx:497) */
WLSQM_API int wlsqm_solver_destroy(wlsqm_solver_t* s);

/* Enqueue the solver's work on a caller-owned CUDA stream (cudaStream_t) instead of its own.  Work already queued on the
 * previous stream is ordered before whatever follows on the new one. */
WLSQM_API int wlsqm_solver_set_stream(wlsqm_solver_t* s, void* cuda_stream);
WLSQM_API int wlsqm_solver_synchronize(wlsqm_solver_t* s);
/* The calling thread's CUDA stream for the entry points WITHOUT a handle (wlsqm_fit_many, wlsqm_interpolate_fit,
 * wlsqm_grid_*, wlsqm_m*): their work runs on it or is ordered after it.  Thread-local; default NULL = the legacy
 * default stream.  A binding that accepts device arrays sets it to the framework's current stream before each call. */
WLSQM_API int wlsqm_set_caller_stream(void* cuda_stream);

/* ExpertSolver.prepare (expert.pyx:309-426) -> expert_prepare_one_{1,2,3}D (expert.pyx:788-817):
 * make_c_*D, make_A, preprocess_A (impl.pyx:70-689).  xi: [ncases][dim] (row stride xi_s0),
 * xk: [ncases][>=nk][dim] (strides xk_s0, xk_s1; 1D: pass dim = 1 with xk_s1 = element stride). */
WLSQM_API int wlsqm_solver_prepare(wlsqm_solver_t* s, const double* xi, int64_t xi_s0, const double* xk, int64_t xk_s0,
                         int64_t xk_s1);

/* ExpertSolver.solve (expert.pyx:467-655) -> impl.solve / solve_iterative (impl.pyx:731-1083).
 * fk [ncases][>=nk] (strides fk_s0, fk_s1); fi [ncases][>=no] in/out (row stride fi_s0): knowns are
 * read, the first no_j entries of row j are written after every case has been solved
 * (expert.pyx:548-557); sens [ncases][>=nk][>=no] (strides sens_s0, sens_s1) or NULL; required if the
 * solver was created with do_sens.  *iters_out (may be NULL) receives the reference's return value:
 * max refinement iterations taken, 0 for ALGO_BASIC. */
WLSQM_API int wlsqm_solver_solve(wlsqm_solver_t* s, const double* fk, int64_t fk_s0, int64_t fk_s1, double* fi,
                       int64_t fi_s0, double* sens, int64_t sens_s0, int64_t sens_s1, int32_t* iters_out);

/* per-case refinement iteration counts of the last ALGO_ITERATIVE solve (host int32[ncases]) */
WLSQM_API int wlsqm_solver_iterations(wlsqm_solver_t* s, int32_t* out);

/* ExpertSolver.interpolate(mode='nearest') with the model index I given
 * (expert_interpolate_nearest, expert.pyx:830-895 -> interpolate_nD, interp.pyx:252-937).
 * x [nx][dim] (row stride x_s0), I int64[nx], diff = a DOF slot index i{1,2,3}_* or WLSQM_DIFF_ALL,
 * out [nx] (or [nx][out_s0] for WLSQM_DIFF_ALL).  Evaluates the solver-owned copy of the last
 * solution, as the reference evaluates Case.fi.  Invalid diff -> WLSQM_E_VALUE. */
WLSQM_API int wlsqm_solver_interpolate(wlsqm_solver_t* s, const double* x, int64_t x_s0, const int64_t* I, int64_t nx,
                             int diff, double* out, int64_t out_s0);

/* ExpertSolver.conds (expert.pyx:429-464): 2-norm condition numbers of the scaled matrices; needs debug. */
WLSQM_API int wlsqm_solver_conds(wlsqm_solver_t* s, double* out);

/* ExpertSolver.memory_used (expert.pyx:289-306): device bytes owned by the solver (used, reserved). */
WLSQM_API int wlsqm_solver_memory(wlsqm_solver_t* s, int64_t* used, int64_t* total);

/* the solver-owned copy of the last solution, [ncases][max no] -> out (row stride out_s0) */
WLSQM_API int wlsqm_solver_get_fi(wlsqm_solver_t* s, double* out, int64_t out_s0);

/* ---- one-shot fits: wlsqm/fitter/simple.pyx:60-604 ------------------------------------------------- */
/* fit_{1,2,3}D[_iterative]_many[_parallel] (generic_fit_*_many*, simple.pyx:731-1170): create +
 * prepare + solve + destroy.  algorithm selects the _iterative variants.  Returns iterations in *iters_out. */
WLSQM_API int wlsqm_fit_many(int dimension, int64_t ncases, const double* xk, int64_t xk_s0, int64_t xk_s1,
                   const double* fk, int64_t fk_s0, int64_t fk_s1, const int32_t* nk, const double* xi,
                   int64_t xi_s0, double* fi, int64_t fi_s0, double* sens, int64_t sens_s0, int64_t sens_s1,
                   int do_sens, const int32_t* order, const int64_t* knowns, const int32_t* weighting_method,
                   int algorithm, int max_iter, int device, int32_t* iters_out);

/* interpolate_fit (interp.pyx:34-143): one model (xi[dim], fi[no]) evaluated at x [nx][dim]. */
WLSQM_API int wlsqm_interpolate_fit(int dimension, int order, const double* xi, const double* fi, const double* x,
                          int64_t x_s0, int64_t nx, int diff, double* out, int device);

/* ---- spatial search on the device (the caller-side cKDTree steps either side of the fitting path) ----------
 * The reference has no such functions: its callers build neighbourhoods with scipy.spatial.cKDTree
 * (examples/expertsolver_example.py:51-66, examples/wlsqm_example.py:100-132) and ExpertSolver searches the
 * nearest / all nearby local models with it (expert.pyx:676-681, 837, 898-911).  These entry points do the same
 * searches on the device (SURVEY.md 8f items 1-3). */
typedef struct wlsqm_grid wlsqm_grid_t;

/* uniform search grid over n points x [n][dim] (row stride x_s0; host or device memory) */
WLSQM_API int wlsqm_grid_create(int dimension, int64_t n, const double* x, int64_t x_s0, int device, wlsqm_grid_t** out);
WLSQM_API int wlsqm_grid_destroy(wlsqm_grid_t* g);
WLSQM_API int wlsqm_grid_info(wlsqm_grid_t* g, int64_t* ncells, double* cell_size, int64_t* bytes);

/* k nearest grid points of every query, ordered by (distance, index) -- cKDTree.query(xq, k).  xq == NULL: the
 * queries are the grid's own points (nq is ignored) and exclude_self drops each point from its own list, i.e.
 * tree.query(x, k+1)[1][:, 1:].  Outputs [nq][k], any of them may be NULL: indices as int32 and/or int64, squared
 * distances.  Missing neighbours (fewer than k points, NaN query) are reported as index n, distance inf. */
WLSQM_API int wlsqm_grid_knn(wlsqm_grid_t* g, const double* xq, int64_t xq_s0, int64_t nq, int k, int exclude_self,
                   int32_t* idx32, int64_t* idx64, double* d2);

/* Fixed-radius neighbourhoods -- cKDTree.query_ball_point(xq, r) (the callers' other neighbourhood search,
 * examples/wlsqm_example.py:100-132), as CSR lists: row q holds the grid points p with
 *     d2(p, q) <= r_q * r_q,   d2 = sum over the axes in axis order of (x_p[d] - q[d])^2,
 * every difference, square, sum and r_q * r_q rounded on its own (no fused multiply-add), identically in every kernel
 * that decides membership.  A point at exactly r is a member (as in cKDTree).
 *   - Points with a NaN or infinite coordinate are never members.  A query with a NaN or infinite coordinate gets an
 *     empty row (cKDTree raises for NaN queries).
 *   - xq == NULL: the queries are the grid's own points (nq is ignored, row i is point i); exclude_self drops only the
 *     point's own index, coincident points stay.  With xq, exclude_self is ignored.
 *   - r: one radius (r_s0 == 0) or one per query (row stride r_s0; for the grid's own points r[i] belongs to point i).
 *     Every radius must be >= 0 and not NaN, else WLSQM_E_VALUE; +inf means every finite point.
 *   - order WLSQM_BALL_BY_INDEX: each row ascending by index (query_ball_point's order for several queries);
 *     WLSQM_BALL_BY_DISTANCE: ascending by (d2, index), the order of wlsqm_grid_knn.
 *   - max_k (0: no cap, else 1..128): a row keeps its max_k members nearest by (d2, index), then arranged by order.
 *     With r = inf, a capped self-query row is the row of wlsqm_grid_knn(k = max_k) as a set, and in the same order
 *     under WLSQM_BALL_BY_DISTANCE, wherever the distances of the row and of the (k+1)-th neighbour are distinct beyond
 *     rounding: wlsqm_grid_knn may fuse the squares and sums of d2 into FMAs, so at near-ties the two can rank
 *     differently.
 * Two calls with the same arguments: the count call gives rowptr int64 [nq + 1] (may be NULL), counts int32 [nq] (may be
 * NULL) and *nnz = rowptr[nq]; the csr call fills col int32 [nnz] for that rowptr (at most 2^31 - 1 entries per call).
 * Any array may be in host or device memory (host ones are staged); the work is ordered after the caller's stream
 * and both calls return when their outputs are written. */
#define WLSQM_BALL_BY_INDEX 0
#define WLSQM_BALL_BY_DISTANCE 1
WLSQM_API int wlsqm_grid_ball_count(wlsqm_grid_t* g, const double* xq, int64_t xq_s0, int64_t nq, const double* r,
                                    int64_t r_s0, int exclude_self, int max_k, int64_t* rowptr, int32_t* counts,
                                    int64_t* nnz);
WLSQM_API int wlsqm_grid_ball_csr(wlsqm_grid_t* g, const double* xq, int64_t xq_s0, int64_t nq, const double* r,
                                  int64_t r_s0, int exclude_self, int max_k, int order, const int64_t* rowptr,
                                  int32_t* col);

/* x[hoods] / f[hoods]: dst[i][k][0..w) = src[idx[i][k]][0..w)  (the caller-side gathers of the examples).
 * src [nsrc][w] (row stride src_s0), idx int32 [n][k] (row stride idx_s0), dst [n][k][w] dense.  Asynchronous on
 * cuda_stream; an index outside [0, nsrc) -- where numpy raises IndexError -- yields NaN, nothing is read out of bounds. */
WLSQM_API int wlsqm_gather_hoods(const double* src, int64_t src_s0, int w, int64_t nsrc, const int32_t* idx, int64_t idx_s0,
                       int64_t n, int k, double* dst, int device, void* cuda_stream);

/* prepare / solve with the neighbourhoods given as index lists (extension): hoods int32 [ncases][>= max nk] into the
 * point array x [npoints][dim] / the per-point data f [npoints]; xk = x[hoods] and fk = f[hoods] are gathered on
 * the device.  xi == NULL: the origins are the first ncases points of x.  solve_hoods takes fi / sens like solve.
 * Only the first nk[i] indices of row i are used (the padding of ragged hoods is never dereferenced); a used index
 * outside [0, npoints) fails with WLSQM_E_VALUE, as x[hoods] raises IndexError in the reference's caller code. */
WLSQM_API int wlsqm_solver_prepare_hoods(wlsqm_solver_t* s, const double* x, int64_t x_s0, int64_t npoints,
                               const int32_t* hoods, int64_t hoods_s0, const double* xi, int64_t xi_s0);
WLSQM_API int wlsqm_solver_solve_hoods(wlsqm_solver_t* s, const double* f, int64_t f_s0, double* fi, int64_t fi_s0,
                             double* sens, int64_t sens_s0, int64_t sens_s1, int32_t* iters_out);

/* Several fields on one geometry in one pass (extension): the operator blocks are streamed once per pass for all fields
 * of the pass instead of once per field (the reference solves each field with its own solve, or with a guest solver).
 * fk [nf][ncases][>= max nk] (strides fk_sf, fk_s0, fk_s1, device arrays fully strided as in wlsqm_solver_solve);
 * fi [nf][ncases][>= max no] in/out (field stride fi_sf, row stride fi_s0, contiguous last axis).  For every field j the
 * unknown slots of fi[j] receive BIT FOR BIT what wlsqm_solver_solve(fk[j], fi[j]) writes on the same solver (same
 * algorithm, kernel path and summation order, ALGO_ITERATIVE refinement with its exact-equality exit per field); known
 * slots and slots >= no_i are not written.  *iters_out (may be NULL) is the maximum of the per-field solve return values;
 * wlsqm_solver_iterations afterwards gives the per-case maximum over the fields.
 *   - The solver's own solution copy is not written: interpolate / get_fi fail with WLSQM_E_NOTREADY until the next
 *     wlsqm_solver_solve (as after keep_solution(0)).
 *   - sens is not produced (it does not depend on the data: take it from one solve or from wlsqm_solver_stencils); a
 *     do_sens solver is accepted.
 *   - WLSQM_E_VALUE: device fk overlapping device fi; an fi layout whose (field, case, slot) map is not injective -- accepted
 *     are fields-outer (fi_sf >= (ncases-1)*fi_s0 + max no, fi_s0 >= max no) and fields-inner (fi_sf >= max no,
 *     fi_s0 >= (nf-1)*fi_sf + max no) with non-negative strides; an active fused gather (wlsqm_solver_set_gather).
 *   - nf = 0 or ncases = 0: no-op, returns 0.  Cases with nr == 0 or nq == 0 behave as in wlsqm_solver_solve.
 *   - Host fk / fi are staged whole (so a host fk aliasing the host fi reads the values from before the call); device
 *     arrays are used in place, asynchronously on the solver's stream.  A guest answers with its host's operators.
 *   - The fields of a pass share the shared-memory ring of the single-field launch shape; nf above what it holds runs
 *     several passes, each streaming the operators again.
 * wlsqm_solver_solve_hoods_fields: the same with the data per point, f [nf][>= npoints] (strides f_sf, f_s0, any), each
 * field equal bit for bit to wlsqm_solver_solve_hoods(f[j], fi[j]); needs prepare_hoods (WLSQM_E_NOTREADY otherwise). */
WLSQM_API int wlsqm_solver_solve_fields(wlsqm_solver_t* s, int64_t nf, const double* fk, int64_t fk_sf, int64_t fk_s0,
                                        int64_t fk_s1, double* fi, int64_t fi_sf, int64_t fi_s0, int32_t* iters_out);
WLSQM_API int wlsqm_solver_solve_hoods_fields(wlsqm_solver_t* s, int64_t nf, const double* f, int64_t f_sf, int64_t f_s0,
                                              double* fi, int64_t fi_sf, int64_t fi_s0, int32_t* iters_out);

/* Export of the prepared operators (extension).  The reference offers the linear map from data to fitted DOFs only
 * as `sens` (impl.pyx:769-779, d fi / d fk, recomputed by every solve), from which its callers assemble Jacobians.
 * Here each of nops operators is a row of coeffs (host memory, [nops][max no], finite, 1 <= nops <= WLSQM_MAXNO): a
 * linear combination of DOF slots.  For case i, with j(s) the reduced index of unknown slot s and t(m) the position of
 * known slot m among the case's knowns (ascending), prepare() stored Op_i (DESIGN.md section 2) and
 *   W[op][i][k] = sum over unknown s < no_i with coeffs[op][s] != 0, ascending s, of coeffs[op][s] * Op_i[k][j(s)]
 *                 (FMA from 0; k < nk_i, 0 beyond),
 *   K[op][i][m] = the same sum over Op_i[nk_i + t(m)][j(s)], plus coeffs[op][m] added last (known m < no_i, 0 elsewhere),
 * so that sum_s coeffs[s] fi[i][s] = sum_k W[i][k] fk[i][k] + sum_m K[i][m] fi_known[i][m] for an ALGO_BASIC solve.
 * The map is the same for ALGO_ITERATIVE solvers (prepare does not depend on the algorithm); the corrections of the
 * refinement loop are not part of it.  Slots >= no_i are ignored; zero coefficients are skipped, never multiplied.
 * A guest answers with its host's operators and neighbour lists.  Outputs are host or device pointers.
 *
 * wlsqm_solver_stencils: W [nops][ncases][max nk], K [nops][ncases][max no] dense (K may be NULL); after any prepare.
 * wlsqm_solver_operator_nnz / _csr: the global sparse operator over the points of prepare_hoods, which must have been
 *   the LAST prepare (WLSQM_E_NOTREADY otherwise).  Row i, column p holds the sum of W[i][k] over k < nk_i with
 *   hoods[i][k] == p, in ascending k.  center = -1: no folding; else 0 <= center, center + ncases <= npoints, and for
 *   every case with slot 0 (F) known, K[i][0] is added last to column center + i and reported as 0 in K ("the known F
 *   of case i is f[center + i]").  Pattern: {(i, hoods[i][k]) : k < nk_i} plus the folded diagonal, columns strictly
 *   ascending, explicit zeros stored; it depends on hoods, knowns and center only and is shared by the nops operators:
 *   rowptr [ncases + 1] and col [nnz] as int32 (index_bits = 32, nnz < 2^31) or int64, values [nops][nnz]. */
WLSQM_API int wlsqm_solver_stencils(wlsqm_solver_t* s, int nops, const double* coeffs, double* W, double* K);
WLSQM_API int wlsqm_solver_operator_nnz(wlsqm_solver_t* s, int64_t center, int64_t* nnz);
WLSQM_API int wlsqm_solver_operator_csr(wlsqm_solver_t* s, int nops, const double* coeffs, int64_t center, int index_bits,
                              void* rowptr, void* col, double* values, double* K);

/* Interpolation operators (extension): the linear map from the data to interpolate(x, mode='nearest', diff) at
 * arbitrary query points, d^D f(xq) = sum_s T_D(s, xq - xi[m]) fi[m][s] with m = I[q] (expert.pyx:687-781).
 * For query q with model m = I[q] and offset h = xq - xi[m], taken per axis:
 *   - per-axis steps are those of steps_of in wlsqm_common.cuh: st = (h, 0.5*h, (1.0/3.0)*h, 0.25*h), each rounded once;
 *   - per-axis Taylor terms: t[0] = 1, t[n] = t[n-1] * st[n-1], with separately rounded multiplies;
 *   - for a slot s with exponents (a, b, c) and a derivative slot D = (p, r, u):
 *       T_D(s) = (tx[a-p] * ty[b-r]) * tz[c-u] if a >= p, b >= r and c >= u;  T_D(s) = 0 otherwise.
 * Coefficient rows keep the convention above ([nops][max no]).  Operator o at query q has the coefficient row
 *   c_q[o][s] = sum over D ascending with coeffs[o][D] != 0 of coeffs[o][D] * T_D(s),
 * each product and each sum rounded separately, with no FMA (__dmul_rn / __dadd_rn: nvcc cannot contract them).
 * Then W, K and the CSR row of query q are EXACTLY the definitions of wlsqm_solver_stencils / _operator_csr for case m
 * with c_q in place of coeffs: the same ascending-slot FMA chain from 0, zero coefficients skipped, c_q[m] added last for
 * known slots, duplicate neighbours merged in ascending k, and with center the known-F weight added last to column
 * center + I[q].  At h = 0, c_q = coeffs: a query at a model origin reproduces that model's stencils / operator row.
 * I[q] outside [0, ncases) (ncases is the search's "none found" for a NaN query): W row 0, K row NaN, empty CSR row,
 * so that W . fk + K . fi is NaN, as interpolate returns NaN for such a query.
 * The operator is the ALGO_BASIC one for every solver (the refinement corrections of ALGO_ITERATIVE are not part of it);
 * it does not read the solver's solution copy (valid after keep_solution(0)).  A guest answers with its host's operators
 * and neighbour lists.  x [nx][dim] (row pitch x_s0) and I (int64 [nx]) may be host or device memory; outputs too.
 *
 * wlsqm_solver_interp_stencils: W [nops][nx][max nk], K [nops][nx][max no] (K may be NULL); valid after ANY prepare.
 * wlsqm_solver_interp_operator_nnz / _csr: rows = queries in caller order, columns = points of prepare_hoods, which
 *   must have been the LAST prepare (WLSQM_E_NOTREADY otherwise); center as for wlsqm_solver_operator_csr; nx = 0 gives
 *   rowptr = [0]. */
WLSQM_API int wlsqm_solver_interp_stencils(wlsqm_solver_t* s, const double* x, int64_t x_s0, const int64_t* I, int64_t nx,
                                           int nops, const double* coeffs, double* W, double* K);
WLSQM_API int wlsqm_solver_interp_operator_nnz(wlsqm_solver_t* s, const int64_t* I, int64_t nx, int64_t center, int64_t* nnz);
WLSQM_API int wlsqm_solver_interp_operator_csr(wlsqm_solver_t* s, const double* x, int64_t x_s0, const int64_t* I, int64_t nx,
                                               int nops, const double* coeffs, int64_t center, int index_bits, void* rowptr,
                                               void* col, double* values, double* K);

/* ExpertSolver.prep_interpolate on the device: index the solver's model origins with a search grid, then
 * interpolate(mode='nearest') may be called with I == NULL, and mode='continuous' is available:
 * weighted average over every model within r, weights (1 - sqrt(d2/r2))^2 (expert.pyx:898-985). */
WLSQM_API int wlsqm_solver_index_models(wlsqm_solver_t* s);
WLSQM_API int wlsqm_solver_nearest_models(wlsqm_solver_t* s, const double* x, int64_t x_s0, int64_t nx, int64_t* I_out);
WLSQM_API int wlsqm_solver_interpolate_continuous(wlsqm_solver_t* s, const double* x, int64_t x_s0, int64_t nx, double r,
                                        int diff, double* out);

/* Continuous-mode interpolation operators (extension): the linear map from the data to interpolate(x, mode='continuous',
 * r, diff), the weighted average of every local model within r (expert.pyx:898-985), as rows per (query, model) pair and
 * as a CSR matrix.  For query q with coordinates x[q]:
 *   - Pairs.  The models of q are the origins xi[m] with d2(xi[m], x[q]) <= r*r under the ball rule of wlsqm_grid_ball_*
 *     (every difference, square and sum rounded on its own, in axis order; the search runs over the solver's model grid
 *     of wlsqm_solver_index_models).  Non-finite origins are never members; a query with a non-finite coordinate has no
 *     models.  The pairs of a query are listed in ascending m -- the rows of cKDTree(xi).query_ball_point(x, r), sorted
 *     -- and numbered query-major: pair_ptr int64 [nx + 1], J int64 [npairs] (the model of each pair).
 *   - Weights.  Per pair, w = tmp * tmp with tmp = 1 - sqrt(d2 / (r*r)), the same rounded d2, every operation rounded on its
 *     own (__ddiv_rn, __dsqrt_rn, __dsub_rn, __dmul_rn); per query S = the sum of w over its pairs in ascending m from +0,
 *     separately rounded adds; alpha = w / S, one rounded division.
 *   - Coefficient rows.  c_q^(m) is the nearest-mode row of wlsqm_solver_interp_stencils at offset h = x[q] - xi[m] (what
 *     it forms for I[q] = m); the pair's row is c_qm[o][s] = alpha * c_q^(m)[o][s], one rounded multiply per entry.  The
 *     pair's W [nops][npairs][max nk] and K [nops][npairs][max no] rows are EXACTLY the definitions of
 *     wlsqm_solver_stencils for case m with c_qm in place of coeffs (ascending-slot FMA chain from 0, zero coefficients
 *     skipped, c_qm[m] added last for known slots).
 *   - CSR row q of E (nx x npoints, columns = points of prepare_hoods) holds, per column p, a sequential sum from +0 in the
 *     order of the row's candidate list: the pairs of q in ascending m; within a pair the neighbours hoods[m][k] in
 *     ascending k, then, with center (as for wlsqm_solver_operator_csr), the pair's known-F weight at column center + m,
 *     which is then reported as 0 in K.  Columns strictly ascending, explicit zeros stored; the pattern depends on x, r,
 *     hoods, knowns and center only and is shared by the nops operators; rowptr / col int32 (index_bits = 32,
 *     nnz < 2^31) or int64, values [nops][nnz].  A row of at most 2048 candidate slots (pairs x (max nk + 1)) is merged
 *     by one warp in shared memory; longer rows are sorted stably by column on the device, over chunks of queries of
 *     bounded scratch, so rows of any length work and the call's total size is not limited.
 * Then  sum_D coeffs[D] d^D f(x[q]) = (E f)[q] + sum over the pairs p of q of K[p] . fi[J[p]]  for an ALGO_BASIC solve, up
 * to rounding against interpolate(x, mode='continuous', r, diff) after the solve.
 *   - A query without a pair has an empty pair range and an empty E row (interpolate returns NaN there).  A query whose
 *     only members lie at exactly r has S = 0 and NaN alpha: its W, K and E entries are NaN (interpolate's 0/0).
 *   - Known difference: wlsqm_solver_interpolate_continuous may contract the sum of d2 into FMAs, so near |x - xi| = r it
 *     can include or exclude a model that the ball rule decides the other way; such a model's weight is below about
 *     2^-100 of a full weight.
 *   - r > 0 (else WLSQM_E_VALUE); the solver must have been indexed (wlsqm_solver_index_models, else WLSQM_E_NOTREADY).
 *   - The map is the ALGO_BASIC one for every solver and does not read the solution copy.  A guest answers with its host's
 *     operators and neighbour lists and with its own model grid, as interpolate does.
 *   - x [nx][dim] (row pitch x_s0) and every output may be host or device memory; host inputs are staged, and the calls
 *     return when their outputs are written.  nx = 0 works (pair_ptr / rowptr = [0]).  One call handles up to 2^31 - 2
 *     pairs (the limit of the ball search); for the CSR one query may hold up to 2^31 - 2 candidate slots and the columns
 *     up to 2^32 - 2 points.
 * wlsqm_solver_interp_continuous_count: pair_ptr (may be NULL), *npairs, and *nnz (may be NULL; counting it needs
 *   prepare_hoods as the last prepare, else WLSQM_E_NOTREADY) for center.
 * wlsqm_solver_interp_continuous_stencils: valid after any prepare; pair_ptr is the count call's for the same x and r
 *   (a different one fails with WLSQM_E_VALUE, so nothing is written past pair_ptr[q + 1]); J [npairs] (may be NULL),
 *   W, K (K may be NULL).
 * wlsqm_solver_interp_continuous_operator_csr: as the stencils call for pair_ptr and J; recounts its pattern (like
 *   wlsqm_solver_operator_csr) and returns rowptr [nx + 1], col, values and K per pair (may be NULL). */
WLSQM_API int wlsqm_solver_interp_continuous_count(wlsqm_solver_t* s, const double* x, int64_t x_s0, int64_t nx, double r,
                                                   int64_t center, int64_t* pair_ptr, int64_t* npairs, int64_t* nnz);
WLSQM_API int wlsqm_solver_interp_continuous_stencils(wlsqm_solver_t* s, const double* x, int64_t x_s0, int64_t nx, double r,
                                                      int nops, const double* coeffs, const int64_t* pair_ptr, int64_t* J,
                                                      double* W, double* K);
WLSQM_API int wlsqm_solver_interp_continuous_operator_csr(wlsqm_solver_t* s, const double* x, int64_t x_s0, int64_t nx,
                                                          double r, int nops, const double* coeffs, int64_t center,
                                                          int index_bits, const int64_t* pair_ptr, int64_t* J, void* rowptr,
                                                          void* col, double* values, double* K);

/* Several fields on one geometry (extension): evaluate caller-held solutions, e.g. the fi written by
 * wlsqm_solver_solve_fields, at query points.  Field j of out is BIT FOR BIT what wlsqm_solver_interpolate (or
 * _interpolate_continuous) writes for the same x, I, diff (and r) when the solver's solution copy holds fi[j][i][0..no_i)
 * for every case i -- what a guest solver answers after its last solve() produced fi[j].  Each query loads its index,
 * coordinates and origin, and in continuous mode walks the model grid, once per pass of up to 8 fields.
 *   - fi [nf][ncases][>= max no], element strides fi_sf, fi_s0 (any non-negative values: it is only read; fields-outer,
 *     fields-inner and fi_sf = 0 all work), contiguous last axis.  Slots >= no_i are never read.
 *   - wlsqm_solver_interpolate_fields (nearest mode): I int64 [nx].  One slot: out[j*out_sf + q*out_sq].
 *     diff == WLSQM_DIFF_ALL: out[j*out_sf + q*out_sq + s] for s < max no, slots >= no_{I[q]} written as 0.0.
 *     I[q] outside [0, ncases) gives NaN, as in wlsqm_solver_interpolate.
 *   - wlsqm_solver_interpolate_continuous_fields: one slot; r > 0 (else WLSQM_E_VALUE); needs wlsqm_solver_index_models
 *     (else WLSQM_E_NOTREADY).  A query with no model within r gives NaN (0/0).
 *   - out: out_sf, out_sq >= 0 in a layout whose (field, query, slot) map is injective, with width 1 or max no:
 *     fields-outer (out_sf >= (nx-1)*out_sq + width, out_sq >= width) or fields-inner (out_sf >= width,
 *     out_sq >= (nf-1)*out_sf + width); else WLSQM_E_VALUE.  A device out overlapping a device fi, x or I: WLSQM_E_VALUE.
 *   - Solver not prepared, or without cases: WLSQM_E_NOTREADY.  Invalid diff: WLSQM_E_VALUE.  nf = 0 or nx = 0: no-op.
 *   - The solver's solution copy is neither read nor written: the calls work after solve_fields and keep_solution(0).
 *   - Any array may be in host or device memory.  Device arrays are used in place, asynchronously on the solver's
 *     stream; host ones are staged, and the call returns when host outputs are written.  A guest answers with its host's
 *     origins. */
WLSQM_API int wlsqm_solver_interpolate_fields(wlsqm_solver_t* s, int64_t nf, const double* fi, int64_t fi_sf, int64_t fi_s0,
                                              const double* x, int64_t x_s0, const int64_t* I, int64_t nx, int diff,
                                              double* out, int64_t out_sf, int64_t out_sq);
WLSQM_API int wlsqm_solver_interpolate_continuous_fields(wlsqm_solver_t* s, int64_t nf, const double* fi, int64_t fi_sf,
                                                         int64_t fi_s0, const double* x, int64_t x_s0, int64_t nx, double r,
                                                         int diff, double* out, int64_t out_sf, int64_t out_sq);

/* The reference keeps the solution twice: in the caller's fi and in each Case (Case_set_fi, infra.pyx:780-786), which is
 * what interpolate() evaluates (expert.pyx:571-699).  A caller that never interpolates can drop the second copy:
 * keep = 0 makes solve() with a device-resident fi write the caller's array only (8 * no bytes per case less traffic);
 * interpolate / get_fi then fail with WLSQM_E_NOTREADY until a solve() with keep = 1.  Default: keep = 1. */
WLSQM_API int wlsqm_solver_keep_solution(wlsqm_solver_t* s, int keep);

/* ---- fused result gather over NVLink peer memory (multi-GPU, one process per GPU) --------------------------------
 * The reference is one process: all cases of a solver write into one fi array (the prange of expert.pyx:536-557).
 * With the cases sharded over GPUs the same array exists once per GPU; instead of an all-gather after the solve, the
 * solve kernel stores every row it computes into ALL copies through peer memory.
 *   wlsqm_peer_alloc: this rank's copy (plain cudaMalloc, zero-filled) and its 64-byte CUDA IPC handle, to be sent to
 *                     the other ranks by any means (torch.distributed.all_gather_object in the Python mirror);
 *   wlsqm_peer_open / _close: map / unmap a peer's copy in this process;  wlsqm_peer_free: release the own copy;
 *   wlsqm_solver_set_gather: row c of this solver is row row0 + c (row stride row_stride >= max no, in doubles) of each
 *                     of the ntargets (<= 8) arrays; ntargets = 0 switches the gather off.
 * Rows written by peers are visible after a synchronisation between the ranks (a stream-ordered barrier per step). */
WLSQM_API int wlsqm_peer_alloc(int device, int64_t bytes, void** ptr, void* ipc_handle_64);
WLSQM_API int wlsqm_peer_open(int device, const void* ipc_handle_64, void** ptr);
WLSQM_API int wlsqm_peer_close(void* ptr);
WLSQM_API int wlsqm_peer_free(void* ptr);
WLSQM_API int wlsqm_solver_set_gather(wlsqm_solver_t* s, int ntargets, void* const* bases, int64_t row0, int64_t row_stride);

/* ---- batched general drivers: wlsqm/utils/lapackdrivers.pyx:1551-1723 ------------------------------ */
/* A (n,n,nlhs) Fortran-contiguous, b (n,nlhs) Fortran, ipiv (n,nlhs) int32 Fortran, 1-based; in place. */
WLSQM_API int wlsqm_mgetrf(int n, int64_t nlhs, double* A, int32_t* ipiv, int device);                 /* mgeneralfactor[p] */
WLSQM_API int wlsqm_mgetrs(int n, int64_t nlhs, const double* LU, const int32_t* ipiv, double* b, int device); /* mgeneralfactored[p] */
WLSQM_API int wlsqm_mgesv(int n, int64_t nlhs, double* A, int32_t* ipiv, double* b, int device);       /* mgeneral[p] */

/* ---- batched symmetric drivers: wlsqm/utils/lapackdrivers.pyx:1107-1354, 204-278 -------------------- */
/* Bunch-Kaufman U D U^T with LAPACK's uplo = 'U' conventions (only the upper triangle of A is read and written; ipiv is
 * dsytrf's: > 0 a 1x1 block, a pair of equal negative entries a 2x2 block).  Same layouts as the general drivers.
 * msytrf = msymmetricfactor[p] (dsytrf, :1199-1233,1275-1314); msytrs = msymmetricfactored[p] (dsytrs, :1236-1272,
 * 1317-1354); msysv = msymmetric[p] (dsysv, :1107-1196; ipiv may be NULL -- the reference discards it);
 * msymmetrize = msymmetrize[p] (A <- (A + A^T)/2, :204-278). */
WLSQM_API int wlsqm_msytrf(int n, int64_t nlhs, double* A, int32_t* ipiv, int device);
WLSQM_API int wlsqm_msytrs(int n, int64_t nlhs, const double* UDU, const int32_t* ipiv, double* b, int device);
WLSQM_API int wlsqm_msysv(int n, int64_t nlhs, double* A, int32_t* ipiv, double* b, int device);
WLSQM_API int wlsqm_msymmetrize(int n, int64_t nlhs, double* A, int device);

/* tridiag (wlsqm/utils/lapackdrivers.pyx:854-877 -> DGTSV, one right-hand side): dl (n-1 used), d (n), du (n-1 used) are
 * overwritten by the factorisation, b by the solution; all four on the host or all four on the device. */
WLSQM_API int wlsqm_gtsv(int n, double* dl, double* d, double* du, double* b, int device);

/* ---- batched matrix equilibration: wlsqm/utils/lapackdrivers.pyx:285-847 --------------------------------------------
 * do_rescale (:319-385) for every matrix of a batch: A (nrows, ncols, nlhs) Fortran-contiguous is scaled in place
 * (apply_scaling_c, :293-299), row_scale (nrows, nlhs) / col_scale (ncols, nlhs) Fortran receive the factors
 * (scaled_b = b * row_scale; x = scaled_x * col_scale).  algo = ScalingAlgo (:305-317): 1 columns (Euclidean), 2 rows,
 * 3 two-pass, 4 Ruiz (2001), 5 SCALGM, 6 DGEEQU.  ok (int32[nlhs], may be NULL): 0 where DGEEQU met a zero row or
 * column -- that matrix is left unscaled (the reference raises LinAlgError for it) -- else 1. */
WLSQM_API int wlsqm_mrescale(int nrows, int ncols, int64_t nlhs, double* A, int algo, double* row_scale, double* col_scale,
                   int32_t* ok, int device);

#ifdef __cplusplus
}
#endif
#endif /* WLSQM_B200_H */
