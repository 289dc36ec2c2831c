// wlsqm_common.cuh -- shared device/host definitions for the wlsqm B200 kernels.
//
// DOF slot tables (exponents of dx,dy,dz per slot) follow the reference's slot order, which is ABI:
//   wlsqm/fitter/defs.pyx:91-103 (1D), :107-133 (2D), :137-183 (3D, irregular order
//   X2,XY,Y2,YZ,Z2,XZ / X3,X2Y,XY2,Y3,Y2Z,YZ2,Z3,XZ2,X2Z,XYZ / X4,...,XYZ2).
// Everything here is written for sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define WLSQM_MAXNO 35          // 3D order 4
#define WLSQM_ALGO_BASIC 1      // defs.pyx:69-70
#define WLSQM_ALGO_ITERATIVE 2
#define WLSQM_WEIGHT_UNIFORM 1  // defs.pyx:74-75
#define WLSQM_WEIGHT_CENTER 2

namespace wlsqm {

// Per-case record (32 B, one aligned load per warp).  Built on the host at solver creation
// (replaces the reference's Case struct, infra.pxd:124-182, and remap(), infra.pyx:145-200).
struct __align__(16) CaseMeta {
    long long op_off;   // offset (in doubles, even) of this case's operator block
    long long knowns;   // bitmask, already restricted to the low `no` bits
    int nk;             // neighbours used by this case
    short no;           // DOFs of the full model
    short nr;           // unknown DOFs = no - popcount(knowns)
    signed char order, wm, nkn, pad0;
    int pad1;
};
static_assert(sizeof(CaseMeta) == 32, "CaseMeta must be 32 bytes");

// exponents (a,b,c) of every DOF slot; 1D and 2D tables are padded with c = 0 / b = c = 0
struct SlotExp { unsigned char a, b, c; };

__host__ __device__ constexpr SlotExp slot_exp_1d(int s) { return SlotExp{(unsigned char)s, 0, 0}; }
__host__ __device__ constexpr SlotExp slot_exp_2d(int s) {
    // order-major, within an order X^(d)Y^0, X^(d-1)Y^1, ..., Y^d
    int d = 0, base = 0;
    while (base + d + 1 <= s) { base += d + 1; ++d; }
    int b = s - base;
    return SlotExp{(unsigned char)(d - b), (unsigned char)b, 0};
}
__host__ __device__ constexpr SlotExp slot_exp_3d(int s) {
    constexpr unsigned char T[35][3] = {
        {0,0,0},
        {1,0,0},{0,1,0},{0,0,1},
        {2,0,0},{1,1,0},{0,2,0},{0,1,1},{0,0,2},{1,0,1},
        {3,0,0},{2,1,0},{1,2,0},{0,3,0},{0,2,1},{0,1,2},{0,0,3},{1,0,2},{2,0,1},{1,1,1},
        {4,0,0},{3,1,0},{2,2,0},{1,3,0},{0,4,0},{0,3,1},{0,2,2},{0,1,3},{0,0,4},{1,0,3},
        {2,0,2},{3,0,1},{2,1,1},{1,2,1},{1,1,2}};
    return SlotExp{T[s][0], T[s][1], T[s][2]};
}
template <int DIM> __host__ __device__ constexpr SlotExp slot_exp(int s) {
    return DIM == 1 ? slot_exp_1d(s) : (DIM == 2 ? slot_exp_2d(s) : slot_exp_3d(s));
}
template <int DIM> __host__ __device__ constexpr int max_no() { return DIM == 1 ? 5 : (DIM == 2 ? 15 : 35); }

__host__ __device__ inline int number_of_dofs(int dim, int order) {   // infra.pyx:67-112
    if (dim < 1 || dim > 3) return -1;
    if (order < 0 || order > 4) return -2;
    const int N[3][5] = {{1,2,3,4,5},{1,3,6,10,15},{1,4,10,20,35}};
    return N[dim-1][order];
}

// the same count in closed form, C(order + DIM, DIM), for kernels: no table lookup in the dependency chain
// index -> order -> number of coefficients -> coefficient loads
template <int DIM> __host__ __device__ constexpr int dofs_of(int order) {
    return DIM == 1 ? order + 1 : (DIM == 2 ? ((order + 1) * (order + 2)) / 2 : ((order + 1) * (order + 2) * (order + 3)) / 6);
}

// ---------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------
#ifdef __CUDACC__

// scaled powers p[a] = d^a / a!  (a = 0..4)
struct Pow5 { double p[5]; };
__device__ __forceinline__ Pow5 scaled_powers(double d) {
    Pow5 r;
    r.p[0] = 1.0; r.p[1] = d; r.p[2] = 0.5 * (d * d);
    r.p[3] = (1.0 / 6.0) * ((d * d) * d);
    r.p[4] = (1.0 / 24.0) * ((d * d) * (d * d));
    return r;
}

// Monomial c^(s) = dx^a dy^b dz^c / (a! b! c!) of slot S (compile-time), from per-axis scaled powers.
// Reference: make_c_{1,2,3}D, wlsqm/fitter/impl.pyx:449-544 / 286-432 / 70-269.
// UNIT0 = true asserts p[0] == 1 on every axis (plain scaled powers) so zero exponents are skipped;
// the derivative evaluator passes shifted tables whose p[0] may be 0 and uses UNIT0 = false.
template <int DIM, int S, bool UNIT0 = true>
__device__ __forceinline__ double monomial(const Pow5& px, const Pow5& py, const Pow5& pz) {
    constexpr SlotExp e = slot_exp<DIM>(S);
    if (!UNIT0) {
        double v = px.p[e.a];
        if (DIM >= 2) v *= py.p[e.b];
        if (DIM >= 3) v *= pz.p[e.c];
        return v;
    }
    double v = px.p[e.a];
    if (DIM >= 2 && e.b > 0) v = (e.a > 0) ? v * py.p[e.b] : py.p[e.b];
    if (DIM >= 3 && e.c > 0) v = (e.a + e.b > 0) ? v * pz.p[e.c] : pz.p[e.c];
    return v;
}

// compile-time loop helper
template <int I, int N, typename F>
__device__ __forceinline__ void static_for(F&& f) {
    if constexpr (I < N) { f(std::integral_constant<int, I>{}); static_for<I + 1, N>(f); }
}

// Model value at offset (dx,dy,dz) from the origin: sum_s fi[s] * monomial_s, highest slots first
// (small terms first).  Same quantity as taylor_{1,2,3}D (wlsqm/fitter/polyeval.pyx:874-948 /
// 550-734 / 82-354), which hard-codes one nested Horner form per (dimension, order); here one
// table-driven sum serves all of them.  `fi` may live in shared or global memory.
template <int DIM>
__device__ __forceinline__ double eval_taylor(int no, const double* __restrict__ fi,
                                              double dx, double dy, double dz) {
    const Pow5 px = scaled_powers(dx);
    const Pow5 py = scaled_powers(DIM >= 2 ? dy : 0.0);
    const Pow5 pz = scaled_powers(DIM >= 3 ? dz : 0.0);
    double acc = 0.0;
    static_for<0, max_no<DIM>()>([&](auto I) {
        constexpr int S = max_no<DIM>() - 1 - decltype(I)::value;
        if (S < no) acc = fma(fi[S], monomial<DIM, S>(px, py, pz), acc);
    });
    return acc;
}

// index of the slot with exponents (a,b,c), or -1 (compile-time search through the slot table)
template <int DIM>
__host__ __device__ constexpr int slot_of(int a, int b, int c) {
    for (int s = 0; s < max_no<DIM>(); ++s) {
        const SlotExp e = slot_exp<DIM>(s);
        if (e.a == a && e.b == b && e.c == c) return s;
    }
    return -1;
}

// f(HI), f(HI-1), ..., f(LO) with compile-time indices (nothing if HI < LO)
template <int HI, int LO, typename F>
__device__ __forceinline__ void static_rfor(F&& f) {
    if constexpr (HI >= LO) { f(std::integral_constant<int, HI>{}); static_rfor<HI - 1, LO>(f); }
}

// h / (t+1), t = 0..3: the factors of the nested form  u0 + h/1 (u1 + h/2 (u2 + h/3 (u3 + h/4 u4)))
struct Steps { double s[4]; };
__device__ __forceinline__ Steps steps_of(double h) { return Steps{{h, 0.5 * h, (1.0 / 3.0) * h, 0.25 * h}}; }

// Value of derivative slot D of the model with coefficients coef(S), S < no: nested Horner form over the
// coefficients with exponents >= those of D.  Only those coefficients are read.  D = 0 is the model value, the
// same nested form as taylor_{1,2,3}D (wlsqm/fitter/polyeval.pyx:874-948 / 550-734 / 82-354).
template <int DIM, int D, typename Coef>
__device__ __forceinline__ double eval_diff_from(Coef&& coef, int no, const Steps& hx, const Steps& hy, const Steps& hz) {
    constexpr SlotExp d = slot_exp<DIM>(D);
    constexpr int p = d.a, q = d.b, r = d.c;
    constexpr int CMAX = DIM >= 3 ? 4 - p - q : 0;
    double vz = 0.0;
    static_rfor<CMAX, r>([&](auto Cc) {
        constexpr int c = decltype(Cc)::value;
        constexpr int BMAX = DIM >= 2 ? 4 - p - c : 0;
        double vy = 0.0;
        static_rfor<BMAX, q>([&](auto Bc) {
            constexpr int b = decltype(Bc)::value;
            constexpr int AMAX = 4 - b - c;
            double vx = 0.0;
            static_rfor<AMAX, p>([&](auto Ac) {
                constexpr int a = decltype(Ac)::value;
                constexpr int S = slot_of<DIM>(a, b, c);
                const double u = S < no ? coef(S) : 0.0;
                if constexpr (a == AMAX) vx = u;
                else vx = fma(vx, hx.s[a - p], u);
            });
            if constexpr (b == BMAX) vy = vx;
            else vy = fma(vy, hy.s[b - q], vx);
        });
        if constexpr (c == CMAX) vz = vy;
        else vz = fma(vz, hz.s[c - r], vy);
    });
    return vz;
}

// coefficients in global memory (read-only path)
template <int DIM, int D>
__device__ __forceinline__ double eval_diff(const double* __restrict__ fg, int no, const Steps& hx, const Steps& hy,
                                            const Steps& hz) {
    return eval_diff_from<DIM, D>([&](int S) { return __ldg(fg + S); }, no, hx, hy, hz);
}

// In-place Taylor shift of the coefficient array along one axis: afterwards u[(a, b, c)] holds the a-th partial
// derivative along AXIS, at offset h (st = steps_of(h)), of the line of coefficients with the other two exponents fixed.
// The interpolation kernels (wlsqm_interp.cu, wlsqm_interp_fields.cu) share it, so their slots agree bit for bit.
template <int DIM, int AXIS>
__device__ __forceinline__ void taylor_shift(double (&u)[max_no<DIM>()], const Steps& st) {
    static_for<0, 5>([&](auto Bc) {
        static_for<0, 5>([&](auto Cc) {
            constexpr int b = decltype(Bc)::value, c = decltype(Cc)::value;   // the other two exponents, in axis order
            constexpr int A = 4 - b - c;
            constexpr bool line = A >= 1 && (DIM >= 3 || c == 0) && (DIM >= 2 || b == 0);
            if constexpr (line) {
                static_for<0, A>([&](auto Jc) {
                    constexpr int j = decltype(Jc)::value;
                    static_rfor<A - 1, j>([&](auto Ic) {
                        constexpr int i = decltype(Ic)::value;
                        constexpr int S0 = AXIS == 0 ? slot_of<DIM>(i, b, c) : (AXIS == 1 ? slot_of<DIM>(b, i, c) : slot_of<DIM>(b, c, i));
                        constexpr int S1 = AXIS == 0 ? slot_of<DIM>(i + 1, b, c) : (AXIS == 1 ? slot_of<DIM>(b, i + 1, c) : slot_of<DIM>(b, c, i + 1));
                        u[S0] = fma(st.s[i], u[S1], u[S0]);
                    });
                });
            }
        });
    });
}
template <int DIM, int AXIS>
__device__ __forceinline__ void taylor_shift(double (&u)[max_no<DIM>()], double h) {
    taylor_shift<DIM, AXIS>(u, steps_of(h));
}

// Model value at offset (dx,dy,dz) from the origin, coefficients anywhere (shared memory in the solve kernel's
// refinement loop): one broadcast load and one FMA per coefficient.
template <int DIM>
__device__ __forceinline__ double eval_taylor_nested(int no, const double* fi, double dx, double dy, double dz) {
    const Steps hx = steps_of(dx), hy = steps_of(DIM >= 2 ? dy : 0.0), hz = steps_of(DIM >= 3 ? dz : 0.0);
    return eval_diff_from<DIM, 0>([&](int S) { return fi[S]; }, no, hx, hy, hz);
}
// ... for a model of the dimension's full size (order 4): no test per coefficient
template <int DIM>
__device__ __forceinline__ double eval_taylor_nested_full(const double* fi, double dx, double dy, double dz) {
    const Steps hx = steps_of(dx), hy = steps_of(DIM >= 2 ? dy : 0.0), hz = steps_of(DIM >= 3 ? dz : 0.0);
    return eval_diff_from<DIM, 0>([&](int S) { return fi[S]; }, max_no<DIM>(), hx, hy, hz);
}

// The same model value at TWO offsets at once (the refinement loop of the solve kernel evaluates the model at a case's
// neighbours, lane = neighbour: with more than 32 neighbours a lane owns two): every coefficient is loaded once for both
// points and the two nested Horner chains are independent, so their latencies overlap.  Same operations per point as
// eval_taylor_nested.
template <int DIM, bool FULL>
__device__ __forceinline__ void eval_taylor_nested2(int no, const double* fi, double dx0, double dy0, double dz0, double dx1,
                                                    double dy1, double dz1, double& r0, double& r1) {
    const Steps hx0 = steps_of(dx0), hy0 = steps_of(DIM >= 2 ? dy0 : 0.0), hz0 = steps_of(DIM >= 3 ? dz0 : 0.0);
    const Steps hx1 = steps_of(dx1), hy1 = steps_of(DIM >= 2 ? dy1 : 0.0), hz1 = steps_of(DIM >= 3 ? dz1 : 0.0);
    constexpr int CMAX = DIM >= 3 ? 4 : 0;
    double vz0 = 0.0, vz1 = 0.0;
    static_rfor<CMAX, 0>([&](auto Cc) {
        constexpr int c = decltype(Cc)::value;
        constexpr int BMAX = DIM >= 2 ? 4 - c : 0;
        double vy0 = 0.0, vy1 = 0.0;
        static_rfor<BMAX, 0>([&](auto Bc) {
            constexpr int b = decltype(Bc)::value;
            constexpr int AMAX = 4 - b - c;
            double vx0 = 0.0, vx1 = 0.0;
            static_rfor<AMAX, 0>([&](auto Ac) {
                constexpr int a = decltype(Ac)::value;
                constexpr int S = slot_of<DIM>(a, b, c);
                const double u = (FULL || S < no) ? fi[S] : 0.0;
                if constexpr (a == AMAX) { vx0 = u; vx1 = u; }
                else { vx0 = fma(vx0, hx0.s[a], u); vx1 = fma(vx1, hx1.s[a], u); }
            });
            if constexpr (b == BMAX) { vy0 = vx0; vy1 = vx1; }
            else { vy0 = fma(vy0, hy0.s[b], vx0); vy1 = fma(vy1, hy1.s[b], vx1); }
        });
        if constexpr (c == CMAX) { vz0 = vy0; vz1 = vy1; }
        else { vz0 = fma(vz0, hz0.s[c], vy0); vz1 = fma(vz1, hz1.s[c], vy1); }
    });
    r0 = vz0;
    r1 = vz1;
}

__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// max over the warp of a non-negative, non-NaN double: its bit pattern orders like an unsigned integer, so
// two REDUX (high word, then low word among the lanes that tie on the high word) replace five shuffle rounds
__device__ __forceinline__ double warp_max_nonneg(double v) {
    const unsigned hi = (unsigned)__double2hiint(v), lo = (unsigned)__double2loint(v);
    const unsigned mh = __reduce_max_sync(0xffffffffu, hi);
    const unsigned ml = __reduce_max_sync(0xffffffffu, hi == mh ? lo : 0u);
    return __hiloint2double((int)mh, (int)ml);
}

// ---- mbarrier + 1D bulk-TMA wrappers (cp.async.bulk, SASS: UBLKCP) ---------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity)
        : "memory");
}
// the same on precomputed 32-bit shared-memory addresses (no generic->shared conversion per use)
__device__ __forceinline__ void mbar_init_u32(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_u32(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait_u32(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(bar), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_1d_u32(uint32_t dst_smem, const void* src_gmem, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
                 "l"(src_gmem), "r"(bytes), "r"(bar)
                 : "memory");
}
// global -> shared bulk copy, completion signalled on `bar` (bytes: multiple of 16, 16B aligned)
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                            uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
// shared -> global bulk store (bulk async-group completion)
__device__ __forceinline__ void tma_store_1d(void* dst_gmem, const void* src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem),
                 "r"(smem_u32(src_smem)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// streaming (evict-first) global accesses for data touched exactly once per pass
__device__ __forceinline__ double ld_stream(const double* p) { return __ldcs(p); }
__device__ __forceinline__ void st_stream(double* p, double v) { __stcs(p, v); }

#endif  // __CUDACC__
}  // namespace wlsqm
