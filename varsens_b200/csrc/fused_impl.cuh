// Fused pipeline: generation + scaling + assembly + objective + estimator reductions in one kernel.
//
// Replaces varsens/saltelli.py:82-125 (Sample), :308-353 (Objective loops) and the reductions of
// :577-622 (Varsens.compute_varsens) for registered functors.  The sample matrices M_1, M_2, N_j,
// N_nj (2*k*n*k*8 bytes in the reference, saltelli.py:119) never exist: a base row i is two
// register vectors A_i, B_i and each of its 2+2k design points is a compile-time selection of
// those registers.
//
// Mapping (one warp = 32 consecutive base rows per batch, persistent grid):
//   phase 1  lane = base row.  A_i, B_i by in-order Halton digit sums (term table in shared
//            memory), scaled; the functor is evaluated on each of the 2+2k points and the value
//            is parked in the warp's shared tile Y[32][M].
//   phase 2  lane = T x T register tile of the symmetric M x M Gram  G += Y^T Y  (M = 2+2k): for
//            each of the 32 rows 2T broadcast shared loads feed T^2 DFMA.  G holds every sum the
//            estimators need (SURVEY.md §3.4).  Shifted sums for var_y stay lane-local in phase 1.
// Warps, then CTAs, are combined in a fixed order -> results are bit-reproducible run to run.
#include <cstdio>
#include <cstdlib>
#include <type_traits>
#include <utility>

#pragma once
#include "device.cuh"

namespace vs {

constexpr int FUSED_WARPS = 8;

__host__ __device__ constexpr uint32_t prime_at(int d) {
    constexpr uint32_t P[32] = {2,  3,  5,  7,  11, 13, 17, 19, 23, 29, 31, 37,  41,  43,  47,  53,
                                59, 61, 67, 71, 73, 79, 83, 89, 97, 101, 103, 107, 109, 113, 127, 131};
    return P[d];
}

__host__ __device__ constexpr int gram_tile_for(int M) {
    int T = 1;
    while (((M + T - 1) / T) * ((M + T - 1) / T + 1) / 2 > 32) ++T;
    return T;
}

// B-point terms of the large bases are computed instead of looked up (see digit_step_arith): dimensions >= AR_D0.
#ifndef VS_ARITH_D0
#define VS_ARITH_D0 11         // prime_at(11) = 37: rows of >= 37 doubles span > 32 banks, random lookups cost 3-5 wavefronts
#endif
constexpr int AR_D0 = VS_ARITH_D0;

template <int K>
struct FusedConst {            // kernel parameter -> constant bank; indexed with compile-time subscripts
    static constexpr int AR_N = K > AR_D0 ? K - AR_D0 : 1;
    double arh[AR_N][HL_J], arl[AR_N][HL_J];   // term of digit at position j of dimension AR_D0 + u = fma(dd, arh, dd * arl), dd = 8 * digit
    double lb[K], wr[K];
    int small_index;           // every Halton index of the run is < 2^29
    int poll_perm;             // see FusedTail::poll_perm
    long long *trace;          // profiling only (VS_TRACE): per-warp clock stamps of CTA 0, else nullptr
    int scale_kind;
};

// Everything the fused kernel does once the CTA partial sums are in HBM (one launch per step): two-level fixed-order combine
// (the last CTA of every group of TAIL_GROUP CTAs sums its group, the last of those sums the groups), packed partial-sum
// vector, optional peer-memory all-reduce over NVLink, estimators, results to device and to mapped host memory.
struct FusedTail {
    double *blockpart;               // [gridDim.x][LROW] compact CTA partial sums
    unsigned *ticket;                // [0] group completion counter, [1 + g] CTA completion counter of group g (reset after use)
    double *partials;                // out: packed partial-sum vector (device) or nullptr
    double *res_dev;                 // out: result vector (device) or nullptr          } mode >= 1
    double *res_host;                // out: result vector + status + time stamps in mapped pinned host memory or nullptr
    double n_total, rows_total;      // divisors of the estimators (saltelli.py:577,591-596; rows < n after NaN trimming)
    int mode;                        // 0 = partial sums only, 1 = + estimators, 2 = + peer exchange + estimators
    int world, rank;
    unsigned epoch;
    const uint64_t *peer_bufs, *peer_flags;     // device arrays [world]: every rank's exchange buffer / flag array as mapped here
    unsigned long long timeout_ns;   // bounded wait for the peers
    double *grouppart;               // [ceil(gridDim.x / TAIL_GROUP)][LROW] second-level partial sums
    int poll_perm;                   // the permutation is being copied into its staging buffer WHILE the kernel runs: entries still
                                     // hold the sentinel 0xFFFFFFFF until their bytes land; every lane polls its own entry and
                                     // puts the sentinel back after reading it (the buffer is clean again when the kernel ends)
};
constexpr int TAIL_GROUP = 16;       // CTAs per first-level combine group
constexpr uint32_t PERM_SENTINEL = 0xFFFFFFFFu;   // never a permutation entry: perm[i] < n <= 2^32 - 1

__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned ld_acquire_sys_u32(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys_u32(unsigned *p, unsigned v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// compile-time loop: fn(std::integral_constant<int, I>{}) for I in [0, N)
template <int N, class Fn, int... I>
__device__ __forceinline__ void static_for_impl(Fn &&fn, std::integer_sequence<int, I...>) {
    (fn(std::integral_constant<int, I>{}), ...);
}
template <int N, class Fn>
__device__ __forceinline__ void static_for(Fn &&fn) {
    static_for_impl<N>(fn, std::make_integer_sequence<int, N>{});
}

template <int N>
__device__ __forceinline__ double tree_product(double (&s)[N]) {
    if constexpr (N == 1) return s[0];
    else {
        constexpr int H = (N + 1) / 2;
        double t[H];
#pragma unroll
        for (int i = 0; i < N / 2; ++i) t[i] = s[2 * i] * s[2 * i + 1];
        if constexpr (N % 2) t[H - 1] = s[N - 1];
        return tree_product<H>(t);
    }
}

// ---- register-resident functors --------------------------------------------------------------
// Every design point is handed to the functor as its own k-vector of registers plus an opaque
// scalar `tok` (value F::token, re-read from shared memory through a volatile load for every
// point).  The functor must fold tok into its first operation on each coordinate.  Without it the
// compiler notices that neighbouring points share k-1 coordinates and hoists the common
// sub-expressions -- i.e. silently applies the separable shortcut -- and the generic path would
// no longer evaluate each point (SURVEY.md §7 "honest flop accounting", §8d).  The token costs one
// LDS per point and no arithmetic.  (Kernel-parameter tokens and register-only tokens were tried: with either,
// ptxas interleaves only 2-3 design points in the evaluation and the kernel gets 10-15 % slower.)
//
// g-function with the division hoisted: prod_c (|4x_c-2| + a_c)/(1+a_c) = C * prod_c (|4x_c-2| + a_c),
// C = prod_c 1/(1+a_c).  Per factor: DFMA (tok*x - 2, tok = 4), DADD (|.| + a_c, a_c from the
// constant bank), DMUL (tree product).
template <int K>
struct GFunctionReg {
    double a[K];
    double C;
    static constexpr bool separable = true;
    static constexpr double token = 4.0;
    __device__ __forceinline__ double factor(int c, double x, double tok) const { return fabs(fma(tok, x, -2.0)) + a[c]; }
    __device__ __forceinline__ double finish(double p) const { return C * p; }
    __device__ __forceinline__ double operator()(const double (&x)[K], double tok) const {
        double s[K];
#pragma unroll
        for (int c = 0; c < K; ++c) s[c] = factor(c, x[c], tok);
        return C * tree_product<K>(s);
    }
};

template <int K>
struct IshigamiReg {
    double A, B;
    static constexpr bool separable = false;
    static constexpr double token = 1.0;
    __device__ __forceinline__ double operator()(const double (&x)[K], double tok) const {
        double s0 = sin(x[0] * tok), s1 = sin(x[1] * tok), x2 = x[2] * tok;
        double x22 = x2 * x2;
        return s0 + A * s1 * s1 + B * (x22 * x22) * s0;
    }
};

// ---- phase 1a: generate + scale the two base points A_i, B_i of the warp's 32 rows (lane = row) ----
// emit(d, A_i[d], B_i[d]) is called once per coordinate, as soon as it is known (a warp that only
// forwards the values to shared memory never holds the 2k-vector in registers).
// Returns whether this lane's row exists (the last batch may be ragged).
template <int K, int SCALE>
__device__ __forceinline__ double scale_coord(const FusedConst<K> &fc, int d, double p) {
    if constexpr (SCALE == VS_SCALE_IDENTITY) return p;
    else return scale_value(SCALE, fc.lb[d], fc.wr[d], p);
}

// ---- Halton digit sums --------------------------------------------------------------------------------------
// Shared-memory copy of the term table in a FIXED layout: dimension d (base b) owns ndmax32(b) rows of b doubles
// at double offset foff(d); row j holds digit / b^(j+1).  Fixed row counts (enough for any 32-bit index) make
// every row address a compile-time immediate of the LDS.  Rows the cached global table does not have are 0.0
// (they are only ever read at digit 0, whose term is 0.0 anyway).
__host__ __device__ constexpr int ndmax32(uint32_t b) {
    int c = 0;
    for (uint64_t m = 0xFFFFFFFFull; m > 0; m /= b) ++c;
    return c;
}
// digits of the largest IB-bit index in base b: the digit positions a run whose indices are all < 2^IB has to visit
template <int IB>
__host__ __device__ constexpr int nd_ib(uint32_t b) {
    int c = 0;
    for (uint64_t m = (IB >= 32 ? 0xFFFFFFFFull : ((1ull << IB) - 1ull)); m > 0; m /= b) ++c;
    return c;
}
__host__ __device__ constexpr uint32_t foff(int d) {          // dimension 0 (base 2) needs no table
    uint32_t s = 0;
    for (int e = 1; e < d; ++e) s += prime_at(e) * (uint32_t)ndmax32(prime_at(e));
    return s;
}
// First digit position from which m * 8b < 2^32 holds for ANY 32-bit index (m_j < 2^32 / b^j): b^(j-1) >= 8.
__host__ __device__ constexpr int jfast(uint32_t b) {
    int j = 1;
    for (uint64_t p = 1; p < 8; p *= b) ++j;
    return j;
}

template <int K>
__device__ __forceinline__ void load_fixed_table(double *__restrict__ dst, const HaltonDev &h, const FusedConst<K> &fc) {
    // the host built the table in this very layout (host.cu: get_halton): one flat, coalesced copy (16 bytes per thread and trip)
    (void)fc;
    constexpr uint32_t N2 = (foff(K) + 1) / 2;
    const double2 *src = reinterpret_cast<const double2 *>(h.fixed);
    for (uint32_t e = threadIdx.x; e < N2; e += blockDim.x) reinterpret_cast<double2 *>(dst)[e] = src[e];
}

// One digit of (m -> m / b, term of m mod b) for two chains.  The in-order additions are __dadd_rn (no
// re-association, no contraction).  FAST form (needs m * 8b < 2^32, proved and brute-forced in
// tools/check_fastdiv.py): c = ceil(2^32 / b);  m*c as a 64-bit product gives q = hi and, from the low word,
// 8*(m mod b) = umulhi(lo, 8b) -- two multiplies, no shift, no subtraction, and the result is already the byte
// offset into the row.  GENERAL form: the compiler's division by a constant.
// Addressing: the term is read with ld.shared [addr + rowoff], rowoff an immediate and addr = 8*(m mod b) + base of the table
// in the shared window.  The base is carried as the HIGH word of a 64-bit addend (`basehi`, kept opaque and live for the
// whole kernel), so that the second multiply delivers the address directly: IMAD.HI(lo, 8b, basehi) = umulhi(lo, 8b) + base.
// (The compiler found that form by itself but re-built the {0, base} register pair with two moves for every step -- 270
// IMAD.MOV per 32 rows in the ncu source view of the first single-launch build, profiles/r02_fused_stalls_by_line.txt.)
// FIRST: the first term initialises the sum (0.0 + t == t for the non-negative table terms; saves a DADD per coordinate).
template <uint32_t B, bool FAST, bool FIRST, uint32_t ROWOFF>
__device__ __forceinline__ void digit_step(uint32_t &m, double &x, uint64_t basehi) {
    double t;
    // The whole step in PTX, so that exactly these instructions come out: IMAD.WIDE (m * c), IMAD.HI with the persistent
    // {0, base} pair as addend (address of the term), LDS with the row offset as immediate, and the DADD.  (Written in C++ the
    // compiler decomposed the 64-bit product, added a uniform zero to the high word and masked low bits of the low word --
    // one or two extra instructions per step.)
    if constexpr (FAST) {
        constexpr uint32_t C = (uint32_t)((0x100000000ull + B - 1) / B);
        asm("{\n\t"
            ".reg .b64 w, a;\n\t"
            ".reg .b32 lo, ah, dm;\n\t"
            "mul.wide.u32 w, %1, %3;\n\t"
            "mov.b64 {lo, %1}, w;\n\t"
            "mul.wide.u32 a, lo, %4;\n\t"
            "add.u64 a, a, %2;\n\t"
            "shr.u64 a, a, 32;\n\t"
            "ld.shared.f64 %0, [a+%5];\n\t"
            "}"
            : "=d"(t), "+r"(m)
            : "l"(basehi), "n"(C), "n"(8u * B), "n"(ROWOFF));
    } else {
        const uint32_t q = m / B;
        const uint32_t addr = (m - q * B) * 8u + (uint32_t)(basehi >> 32);
        m = q;
        asm("ld.shared.f64 %0, [%1+%2];" : "=d"(t) : "l"((uint64_t)addr), "n"(ROWOFF));
    }
    if constexpr (FIRST) x = t;
    else x = __dadd_rn(x, t);
}

// The same step with the term COMPUTED instead of looked up (B-points of bases >= 37, whose table rows span more than the
// 32 banks: a random 8-byte lookup costs 3-5 shared-memory wavefronts, and generation is bound by that SM-wide pipe while
// the FP64 pipe idles).  With dd = 8 * digit exact in fp64 (magic-number conversion, one DADD) the term digit / b^(j+1) is
//   fma(dd, rh, dd * rl),   rh = RN(1 / b^(j+1)) / 8,  rl = RN(1 / b^(j+1) - RN(1 / b^(j+1))) / 8
// i.e. the product of dd with a double-double reciprocal, rounded once.  Its error before the final rounding is < 2^-104
// relative, while digit / b^(j+1) (odd denominator) stays >= 2^-85 relative away from every rounding boundary, so the
// result IS the correctly rounded quotient; on top of the argument the host compares all digits of all positions against
// the term table when the constants are built (host.cu: build_arith) and refuses the fused kernel on any mismatch.
// The other term-table modes use rl = 0 and rh = their factor: the same instruction sequence gives RN(digit * factor).
template <uint32_t B, bool FAST, bool FIRST>
__device__ __forceinline__ void digit_step_arith(uint32_t &m, double &x, double rh, double rl) {
    uint32_t off8;
    if constexpr (FAST) {
        constexpr uint32_t C = (uint32_t)((0x100000000ull + B - 1) / B);
        const uint64_t w = (uint64_t)m * C;
        off8 = __umulhi((uint32_t)w, 8u * B);
        m = (uint32_t)(w >> 32);
    } else {
        const uint32_t q = m / B;
        off8 = (m - q * B) * 8u;
        m = q;
    }
    const double dd = __dadd_rn(__hiloint2double(0x43300000, (int)off8), -4503599627370496.0);
    const double t = __fma_rn(dd, rh, __dmul_rn(dd, rl));
    if constexpr (FIRST) x = t;
    else x = __dadd_rn(x, t);
}

// Halton digit sums of the two indices ia (A_i) and ib (B_i) for one GROUP of HG dimensions: 2*HG independent
// (index, sum) chains advance together, least-significant digit first; the group stops after the largest digit
// count it needs for this run (warp-uniform).  Group 0 also emits dimension 0: base 2, where every partial sum
// is exact and the in-order digit sum is a bit reversal.
#ifndef VS_HG
#define VS_HG 4
#endif
constexpr int HG = VS_HG;
template <int K>
__host__ __device__ constexpr int halton_groups() { return K > 1 ? (K - 1 + HG - 1) / HG : 1; }

template <int K, int SCALE, int G, int IB, class Emit>
__device__ __forceinline__ void halton_group(const FusedConst<K> &fc, uint64_t basehi, uint32_t ia, uint32_t ib, Emit &&emit) {
    if constexpr (G == 0)
        emit(0, scale_coord<K, SCALE>(fc, 0, (double)__brev(ia) * 2.3283064365386962890625e-10),
             scale_coord<K, SCALE>(fc, 0, (double)__brev(ib) * 2.3283064365386962890625e-10));
    constexpr int D0 = 1 + G * HG;
    if constexpr (D0 < K) {
        constexpr int N = (K - D0) < HG ? (K - D0) : HG;
        constexpr int JMAX = nd_ib<IB>(prime_at(D0));       // the smallest base of the group has the most digits
        uint32_t ma[N], mb[N];
        double xa[N], xb[N];
#pragma unroll
        for (int u = 0; u < N; ++u) {
            ma[u] = ia;
            mb[u] = ib;
            xa[u] = 0.0;
            xb[u] = 0.0;
        }
        const bool small = IB <= 29 || fc.small_index != 0; // every index of the run < 2^29: FAST from digit 1 on
        // All digit positions an IB-bit index can have are executed unconditionally: one straight-line block per group, so
        // the scheduler can run the index chains ahead and keep many table loads in flight (with a branch per digit the
        // loads of digit j+1 could not be hoisted over the additions of digit j and every digit paid a full, queue-inflated
        // LDS latency).  Positions beyond a run's digit count see m == 0 and add +0.0 (exact).  IB is a template parameter
        // (26 or 32): BASELINE's configs all stay below 2^26 and visit 132 instead of 159 positions per point at k = 20.
        static_for<JMAX>([&](auto Jc) {
            constexpr int J = decltype(Jc)::value;
            {
                static_for<N>([&](auto Uc) {
                    constexpr int U = decltype(Uc)::value;
                    constexpr uint32_t B = prime_at(D0 + U);
                    if constexpr (J < nd_ib<IB>(B)) {
                        constexpr uint32_t RO = (uint32_t)(foff(D0 + U) + J * B) * 8u;   // byte offset of the row inside the table
                        constexpr bool AR = (D0 + U) >= AR_D0;               // B-point term computed, not looked up
                        constexpr int AU = AR ? (D0 + U - AR_D0) : 0, AJ = J < HL_J ? J : HL_J - 1;
                        constexpr bool F1 = J == 0;
                        if constexpr (J == 0 && !(IB <= 29 && 8ull * B * ((1ull << (IB < 32 ? IB : 31))) <= 0x100000000ull)) {
                            digit_step<B, false, F1, RO>(ma[U], xa[U], basehi);
                            if constexpr (AR) digit_step_arith<B, false, F1>(mb[U], xb[U], fc.arh[AU][AJ], fc.arl[AU][AJ]);
                            else digit_step<B, false, F1, RO>(mb[U], xb[U], basehi);
                        } else if constexpr (J == 0 || J >= jfast(B) || IB <= 29) {
                            digit_step<B, true, F1, RO>(ma[U], xa[U], basehi);
                            if constexpr (AR) digit_step_arith<B, true, F1>(mb[U], xb[U], fc.arh[AU][AJ], fc.arl[AU][AJ]);
                            else digit_step<B, true, F1, RO>(mb[U], xb[U], basehi);
                        } else if (small) {
                            digit_step<B, true, F1, RO>(ma[U], xa[U], basehi);
                            if constexpr (AR) digit_step_arith<B, true, F1>(mb[U], xb[U], fc.arh[AU][AJ], fc.arl[AU][AJ]);
                            else digit_step<B, true, F1, RO>(mb[U], xb[U], basehi);
                        } else {
                            digit_step<B, false, F1, RO>(ma[U], xa[U], basehi);
                            if constexpr (AR) digit_step_arith<B, false, F1>(mb[U], xb[U], fc.arh[AU][AJ], fc.arl[AU][AJ]);
                            else digit_step<B, false, F1, RO>(mb[U], xb[U], basehi);
                        }
                    }
                });
            }
        });
#pragma unroll
        for (int u = 0; u < N; ++u) emit(D0 + u, scale_coord<K, SCALE>(fc, D0 + u, xa[u]), scale_coord<K, SCALE>(fc, D0 + u, xb[u]));
    }
}

template <int K, int SCALE, int IB, class Emit>
__device__ __forceinline__ bool gen_rows_impl(const SourceDev &src, const FusedConst<K> &fc, uint64_t basehi, uint64_t i_begin,
                                              uint64_t rows, uint64_t bt, int lane, Emit &&emit) {
    uint64_t r = bt * 32 + lane;
    const bool valid = r < rows;
    const uint64_t i = i_begin + (valid ? r : rows - 1);
    uint64_t pi;
    if (fc.poll_perm) {
        // host permutation still on its way (one cudaMemcpyAsync enqueued before this launch): wait for my own entry
        uint32_t v = 0u;
        if (valid) {
            uint32_t *pp = const_cast<uint32_t *>(src.perm) + i;
            for (;;) {
                asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(pp) : "memory");
                if (v != PERM_SENTINEL) break;
                __nanosleep(100);
            }
            *pp = PERM_SENTINEL;                          // leave the staging buffer clean for the next call
        }
        pi = v;
    } else {
        pi = src.perm[i];
    }
    if (src.raw) {
        const double *ra = src.raw + i * (uint64_t)K, *rb = src.raw + (src.n + pi) * (uint64_t)K;
#pragma unroll
        for (int d = 0; d < K; ++d) emit(d, scale_coord<K, SCALE>(fc, d, ra[d]), scale_coord<K, SCALE>(fc, d, rb[d]));
    } else {
        const uint32_t ia = (uint32_t)(src.start + i), ib = (uint32_t)(src.start + src.n + pi);
        static_for<halton_groups<K>()>([&](auto Gc) { halton_group<K, SCALE, decltype(Gc)::value, IB>(fc, basehi, ia, ib, emit); });
    }
    return valid;
}

// One warp-uniform branch on the scale kind for the whole row (not one per coordinate).
template <int K, int IB = 32, class Emit>
__device__ __forceinline__ bool gen_rows(const SourceDev &src, const FusedConst<K> &fc, uint64_t basehi, uint64_t i_begin, uint64_t rows,
                                         uint64_t bt, int lane, Emit &&emit) {
    if (fc.scale_kind == VS_SCALE_IDENTITY) return gen_rows_impl<K, VS_SCALE_IDENTITY, IB>(src, fc, basehi, i_begin, rows, bt, lane, emit);
    if (fc.scale_kind == VS_SCALE_LINEAR) return gen_rows_impl<K, VS_SCALE_LINEAR, IB>(src, fc, basehi, i_begin, rows, bt, lane, emit);
    return gen_rows_impl<K, VS_SCALE_POWER, IB>(src, fc, basehi, i_begin, rows, bt, lane, emit);
}

// {0, shared-window address of the term table} as one opaque 64-bit value (see digit_step)
__device__ __forceinline__ uint64_t table_basehi(const double *terms) {
    uint64_t v = (uint64_t)(uint32_t)__cvta_generic_to_shared(terms) << 32;
    asm volatile("" : "+l"(v));
    return v;
}

// Generic evaluation of EG design points of one base row for a product-form functor (see eval_rows).
#ifndef VS_EG
#define VS_EG 12
#endif
constexpr int EG = VS_EG;
template <int K>
__host__ __device__ constexpr int eval_groups() { return (2 + 2 * K + EG - 1) / EG; }

// ---- paired tile layout ------------------------------------------------------------------------------------------
// The second-order estimators read the J/N blocks of the Gram only in the symmetric combinations
//   N_i.N_j + J_i.J_j  (saltelli.py:618-619)   and   N_i.J_j + J_i.N_j  (:612-613),      J_j = f(N_j[j]), N_j = f(N_nj[j]),
// and with P = N + J, M = N - J these are (P_i.P_j + M_i.M_j)/2 and (P_i.P_j - M_i.M_j)/2; the first-order sums follow from
// A.P_j, A.M_j, B.P_j, B.M_j.  So instead of the Gram of the (2+2K)-vector (A, B, J, N) the S-warps accumulate the Grams
// of the two (K+2)-vectors  w = (P_0..P_{K-1}, A, B)  and  u = (M_0..M_{K-1}, A, B):  2 * HB(HB+1)/2 8x8 tiles with
// HB = ceil((K+2)/8) instead of NB(NB+1)/2 with NB = ceil((2+2K)/8) -- 12 instead of 21 DMMA per 4 rows at K = 20.
// The E-warp forms P_j, M_j when both members of a pair are evaluated (2 extra DADD per pair); pm_scatter_kernel maps
// the CTA sums back to the packed partial-sum vector (second-order blocks symmetrised, see include/varsens_b200.h).
template <int K> __host__ __device__ constexpr int pm_hb() { return (K + 2 + 7) / 8; }
template <int K> __host__ __device__ constexpr bool pm_pays() {
    constexpr int nb = (2 + 2 * K + 7) / 8, hb = (K + 2 + 7) / 8;
    return hb * (hb + 1) < nb * (nb + 1) / 2;
}

// Evaluation slot E -> design point.  Plain order: E = p.  Paired order: A, B, then (N_j[j], N_nj[j]) for j = 0, 1, ...
template <int K, bool PM> __host__ __device__ constexpr int point_of_slot(int E) {
    return (!PM || E < 2) ? E : (((E - 2) & 1) ? 2 + K + (E - 2) / 2 : 2 + (E - 2) / 2);
}

template <int K, class F, int G, bool PM, class YR>
__device__ __forceinline__ void eval_group(const F &f, const double (&tk)[EG], const double (&a)[K], const double (&b)[K], bool valid,
                                           const YR &Yrow, double &fA, double &fB) {
    static_assert(!PM || EG % 2 == 0, "paired layout needs both members of a pair in one evaluation group");
    constexpr int M = 2 + 2 * K;
    constexpr int P0 = G * EG;
    constexpr int NP = (M - P0) < EG ? (M - P0) : EG;
    constexpr int HS = 8 * pm_hb<K>();
    double pr[NP] = {};
    static_for<K>([&](auto Cc) {
        constexpr int C = decltype(Cc)::value;
        static_for<NP>([&](auto Uc) {
            constexpr int U = decltype(Uc)::value;
            constexpr int P = point_of_slot<K, PM>(P0 + U);
            // point P: 0 = A_i, 1 = B_i, 2+J = B_i with column J from A_i, 2+K+J = A_i with column J from B_i
            constexpr bool fromA = (P == 0) || (P >= 2 && P < 2 + K && C == P - 2) || (P >= 2 + K && C != P - 2 - K);
            const double s_ = f.factor(C, fromA ? a[C] : b[C], tk[U]);
            pr[U] = (C == 0) ? s_ : pr[U] * s_;
        });
    });
    static_for<NP>([&](auto Uc) {
        constexpr int U = decltype(Uc)::value;
        constexpr int P = point_of_slot<K, PM>(P0 + U);
        if constexpr (P == 0) fA = f.finish(pr[U]);
        else if constexpr (P == 1) fB = f.finish(pr[U]);
        else if constexpr (!PM) Yrow[P] = valid ? f.finish(pr[U]) : 0.0;
        else if constexpr (P >= 2 + K) {                           // second member of pair j: slot U-1 holds f(N_j[j])
            constexpr int J = P - 2 - K;
            const double vj = f.finish(pr[U - 1]), vn = f.finish(pr[U]);
            Yrow[J] = valid ? vn + vj : 0.0;
            Yrow[HS + J] = valid ? vn - vj : 0.0;
        }
    });
}

struct YRef {                                  // value p of a lane's row lives at p[i * st]
    double *p;
    int st;
    __device__ __forceinline__ double &operator[](int i) const { return p[i * st]; }
};

// ---- phase 1b: evaluate the functor on the 2+2k points of the lane's row; values go to Yrow ----
template <int K, class F, bool SEPARABLE, bool PM = false>
__device__ __forceinline__ void eval_rows(const F &f, volatile double *tokp, const double (&a)[K], const double (&b)[K],
                                          bool valid, double *__restrict__ Ybase, double shift, double &sA, double &qA,
                                          double &sB, double &qB, const int ystride = 1) {
    // value p of this lane's row lives at Ybase[p * ystride] (row-major tile: stride 1; p-major tile: stride = pitch)
    const YRef Yrow{Ybase, ystride};
    double fA, fB;
    if constexpr (SEPARABLE && F::separable) {
        // product-form shortcut: all 2+2k values from prefix/suffix products of the 2k factors
        // (O(k) per row instead of O(k^2)).  Prefix pass parks prefix*factor in the tile, suffix
        // pass completes it in place -- no k-long register arrays besides the factors.
        double ga[K], gb[K];
#pragma unroll
        for (int c = 0; c < K; ++c) { ga[c] = f.factor(c, a[c], F::token); gb[c] = f.factor(c, b[c], F::token); }
        double pa = 1.0, pb = 1.0;
#pragma unroll
        for (int j = 0; j < K; ++j) {
            Yrow[2 + j] = pb * ga[j];                            // N_j[j]  = B with column j from A
            Yrow[2 + K + j] = pa * gb[j];                        // N_nj[j] = A with column j from B
            pa *= ga[j];
            pb *= gb[j];
        }
        fA = f.finish(pa);
        fB = f.finish(pb);
        double sa = f.finish(1.0), sb = f.finish(1.0);           // suffix products carry the constant C
#pragma unroll
        for (int j = K - 1; j >= 0; --j) {
            double vj = Yrow[2 + j] * sb, vn = Yrow[2 + K + j] * sa;
            Yrow[2 + j] = valid ? vj : 0.0;
            Yrow[2 + K + j] = valid ? vn : 0.0;
            sa *= ga[j];
            sb *= gb[j];
        }
    } else if constexpr (F::separable) {
        // Generic path for product-form functors: every factor of every point is evaluated (no sharing between
        // points -- each point has its own opaque token), but EG points advance together, factor by factor, each
        // with a running product (EG = 12 measured best: 8 -> 5.4 ms, 12 -> 5.2 ms).  That gives the scheduler EG independent DMUL chains plus 2*EG independent
        // DFMA/DADD per step (FP64 latency covered inside one warp) and needs no k-long temporary arrays.
        fA = 0.0;
        fB = 0.0;
        static_for<eval_groups<K>()>([&](auto Gc) {
            double tk[EG];
#pragma unroll
            for (int u = 0; u < EG; ++u) tk[u] = *tokp;
            eval_group<K, F, decltype(Gc)::value, PM>(f, tk, a, b, valid, Yrow, fA, fB);
        });
    } else {
        static_assert(!PM, "paired layout is implemented for product-form functors");
        fA = f(a, *tokp);
        fB = f(b, *tokp);
        static_for<K>([&](auto Jc) {
            constexpr int J = decltype(Jc)::value;
            double xj[K], xn[K];
#pragma unroll
            for (int c = 0; c < K; ++c) {
                xj[c] = (c == J) ? a[c] : b[c];                  // N_j[J]   (saltelli.py:119-123)
                xn[c] = (c == J) ? b[c] : a[c];                  // N_nj[J]
            }
            double vj = f(xj, *tokp), vn = f(xn, *tokp);
            Yrow[2 + J] = valid ? vj : 0.0;
            Yrow[2 + K + J] = valid ? vn : 0.0;
        });
    }
    if constexpr (PM) {
        static_assert(!(SEPARABLE && F::separable), "the prefix/suffix shortcut keeps the plain layout");
        constexpr int HS = 8 * pm_hb<K>();
        Yrow[K] = Yrow[HS + K] = valid ? fA : 0.0;
        Yrow[K + 1] = Yrow[HS + K + 1] = valid ? fB : 0.0;
    } else {
        Yrow[0] = valid ? fA : 0.0;
        Yrow[1] = valid ? fB : 0.0;
    }
    if (valid) {
        double dA = fA - shift, dB = fB - shift;
        sA += dA;
        qA = fma(dA, dA, qA);
        sB += dB;
        qB = fma(dB, dB, qB);
    }
}

template <int K, class F, bool SEPARABLE>
__device__ __forceinline__ void rows_phase(const SourceDev &src, const FusedConst<K> &fc, const F &f,
                                           const double *__restrict__ terms, volatile double *tokp, uint64_t i_begin,
                                           uint64_t rows, uint64_t bt, int lane, double *__restrict__ Yrow, double shift,
                                           double &sA, double &qA, double &sB, double &qB) {
    double a[K], b[K];
    const bool valid = gen_rows<K>(src, fc, table_basehi(terms), i_begin, rows, bt, lane, [&](int d, double xa, double xb) {
        a[d] = xa;
        b[d] = xb;
    });
    eval_rows<K, F, SEPARABLE>(f, tokp, a, b, valid, Yrow, shift, sA, qA, sB, qB);
}

template <int K, class F, bool SECOND, bool SEPARABLE>
__global__ void __launch_bounds__(FUSED_WARPS * 32, 1)
fused_kernel(SourceDev src, FusedConst<K> fc, F f, uint64_t i_begin, uint64_t i_end, const double *__restrict__ shift_ptr,
             double *__restrict__ blockpart) {
    constexpr int M = 2 + 2 * K;
    constexpr int T = SECOND ? gram_tile_for(M) : 2;
    constexpr int NT = (M + T - 1) / T;
    constexpr int MP = (NT * T) % 2 ? NT * T : NT * T + 1;     // odd row pitch
    constexpr int NTILES = SECOND ? NT * (NT + 1) / 2 : NT;    // first-order only: tile row 0 (fM_1, fM_2) x all columns
    static_assert(SECOND ? NTILES <= 32 : true, "Gram does not fit one tile per lane");
    constexpr int TPL = SECOND ? 1 : (NTILES + 31) / 32;

    extern __shared__ double smem[];
    double *terms = smem;                                           // shared copy of the Halton term table
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t nterms = src.raw ? 0u : ((foff(K) + 1u) & ~1u);     // even: the table is copied 16 bytes at a time
    volatile double *tokp = smem + nterms;                          // opaque functor token (see the functors)
    double *Y = smem + nterms + 1 + (size_t)warp * 32 * MP;         // this warp's [32][MP] value tile
    if (nterms) load_fixed_table<K>(terms, src.h, fc);
    if (threadIdx.x == 0) *tokp = F::token;
    // zero the padding columns once (never written again)
    for (int e = lane; e < 32 * (MP - M); e += 32) Y[(e / (MP - M)) * MP + M + e % (MP - M)] = 0.0;
    __syncthreads();

    const double shift = *shift_ptr;
    double sA = 0.0, qA = 0.0, sB = 0.0, qB = 0.0;
    double acc[TPL][T][T];
#pragma unroll
    for (int q = 0; q < TPL; ++q)
#pragma unroll
        for (int x = 0; x < T; ++x)
#pragma unroll
            for (int y = 0; y < T; ++y) acc[q][x][y] = 0.0;
    int tr[TPL], tc[TPL];
#pragma unroll
    for (int q = 0; q < TPL; ++q) {
        int id = lane + 32 * q;
        if (SECOND) tile_coords(id < NTILES ? id : 0, NT, tr[q], tc[q]);
        else { tr[q] = 0; tc[q] = id < NTILES ? id : 0; }
    }

    const uint64_t rows = i_end - i_begin;
    const uint64_t nbatch = (rows + 31) / 32;
    const uint64_t wstride = (uint64_t)gridDim.x * FUSED_WARPS;
    for (uint64_t bt = (uint64_t)blockIdx.x * FUSED_WARPS + warp; bt < nbatch; bt += wstride) {
        rows_phase<K, F, SEPARABLE>(src, fc, f, terms, tokp, i_begin, rows, bt, lane, Y + lane * MP, shift, sA, qA, sB, qB);
        __syncwarp();
        // ------------------------------ phase 2: lane = Gram tile ------------------------------
#pragma unroll 4
        for (int rr = 0; rr < 32; ++rr) {
            const double *row = Y + rr * MP;
#pragma unroll
            for (int q = 0; q < TPL; ++q) {
                double ta[T], tb[T];
#pragma unroll
                for (int x = 0; x < T; ++x) { ta[x] = row[tr[q] * T + x]; tb[x] = row[tc[q] * T + x]; }
                if constexpr (SECOND) {
#pragma unroll
                    for (int x = 0; x < T; ++x)
#pragma unroll
                        for (int y = 0; y < T; ++y) acc[q][x][y] = fma(ta[x], tb[y], acc[q][x][y]);
                } else {
#pragma unroll
                    for (int x = 0; x < 2; ++x)                       // rows fM_1, fM_2 only (T == 2)
#pragma unroll
                        for (int y = 0; y < T; ++y) acc[q][x][y] = fma(ta[x], tb[y], acc[q][x][y]);
                }
            }
        }
        __syncwarp();
    }

    // ---- combine warps in warp order through shared memory, then write this CTA's partial ----
    __syncthreads();
    constexpr int TT = T * T;
    double *red = smem;                                   // [TPL*32][TT] + 4
    sA = warp_sum(sA); qA = warp_sum(qA); sB = warp_sum(sB); qB = warp_sum(qB);
    for (int w = 0; w < FUSED_WARPS; ++w) {
        if (warp == w) {
#pragma unroll
            for (int q = 0; q < TPL; ++q)
#pragma unroll
                for (int x = 0; x < T; ++x)
#pragma unroll
                    for (int y = 0; y < T; ++y) {
                        double *p = red + ((size_t)(q * 32 + lane)) * TT + x * T + y;
                        *p = (w == 0) ? acc[q][x][y] : *p + acc[q][x][y];
                    }
            if (lane == 0) {
                double *s4 = red + (size_t)TPL * 32 * TT;
                if (w == 0) { s4[0] = sA; s4[1] = sB; s4[2] = qA; s4[3] = qB; }
                else { s4[0] += sA; s4[1] += sB; s4[2] += qA; s4[3] += qB; }
            }
        }
        __syncthreads();
    }
    constexpr int PER_BLOCK = TPL * 32 * TT + 4;
    for (int e = threadIdx.x; e < PER_BLOCK; e += blockDim.x) blockpart[(size_t)blockIdx.x * PER_BLOCK + e] = red[e];
}


// ---------------------------------------------------------------------------------------------
// Warp specialisation helpers.  E-warps run phase 1 only (generation + evaluation, no Gram
// accumulators -> more warps per SM); S-warps run the Gram update only.  S-warp s serves the E-warps
// with the same warp id mod 4, i.e. the ones that share its SM sub-partition and FP64 pipe.  Tiles
// are handed over through full/empty mbarrier pairs (producer: __syncwarp + one arrive; consumer:
// try_wait.parity); there is no CTA-wide barrier inside the loop.
// ---------------------------------------------------------------------------------------------
constexpr int WS_S = 4;                       // one S-warp per SM sub-partition

// ---------------------------------------------------------------------------------------------
// Two-role variant with the Gram update on the FP64 tensor path (DMMA, mma.sync m8n8k4.f64).
// Measured on B200 (profiles/r01_fp64_pipes_microbench.txt): DMMA and DFMA share one 36-37 TFLOP/s
// FP64 datapath, so DMMA adds no flops -- what it removes is shared-memory traffic and issue slots:
// the register-tile SYRK needs 12 LDS.64 per row per lane (768 wavefronts per 32-row batch, and the
// LSU pipe is shared by the four sub-partitions), the tensor path needs 6 fragment loads per FOUR
// rows (96 wavefronts per batch) and 168 instead of 1152 issue slots.
//   Y tile is p-major here: Yt[p][row] with pitch 36 -> E-warp stores are unit-stride, and the
//   fragment  f_P = Yt[8P + lane/4][r0 + lane%4]  is both the A (row) and the B (col) operand of
//   G[P][Q] += Y[r0..r0+4, P]^T Y[r0..r0+4, Q]  and loads conflict-free in two wavefronts.
//   M is padded to NB = ceil(M/8) blocks (rows M..8NB-1 of the tile stay zero).
// ---------------------------------------------------------------------------------------------
constexpr int YT_PITCH = 36;

template <int K, class F, bool SEPARABLE>
__host__ __device__ constexpr bool wsd_paired() { return pm_pays<K>() && F::separable && !SEPARABLE; }

// Upper-triangular tile walk shared by the S-warp update, the combine step and nothing else: fn(t, P, Q) with block
// coordinates inside the padded tile row (paired layout: two independent triangles).
template <int NB, int HB, bool PM, class Fn>
__device__ __forceinline__ void for_each_tile(Fn &&fn) {
    int t = 0;
    if constexpr (PM) {
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int P = 0; P < HB; ++P)
#pragma unroll
                for (int Q = P; Q < HB; ++Q, ++t) fn(t, h * HB + P, h * HB + Q);
    } else {
#pragma unroll
        for (int P = 0; P < NB; ++P)
#pragma unroll
            for (int Q = P; Q < NB; ++Q, ++t) fn(t, P, Q);
    }
}

// ---- compact CTA partial sums and the last-CTA tail ---------------------------------------------------------------
// A CTA's partial sums are stored tile-major: tile t of the for_each_tile walk owns 64 doubles, the C fragment of lane L
// (row L/4, columns 2(L%4), 2(L%4)+1 of the 8x8 tile) at [t*64 + 2L, +1]; then the four shifted sums; padded to LROW.
template <int NB, int HB, bool PM>
__host__ __device__ constexpr int wsd_ntl() { return PM ? HB * (HB + 1) : NB * (NB + 1) / 2; }
template <int NB, int HB, bool PM>
__host__ __device__ constexpr int wsd_lrow() { return wsd_ntl<NB, HB, PM>() * 64 + 8; }

// dense entry (x, y) (padded coordinates, either order) of the combined CTA sums D
template <int NB, int HB, bool PM>
__device__ __forceinline__ double dense_at(const double *__restrict__ D, int x, int y) {
    const int lo = x < y ? x : y, hi = x < y ? y : x;
    int P = lo >> 3, Q = hi >> 3, t;
    if constexpr (PM) {
        const int h = P / HB;
        P -= h * HB;
        Q -= h * HB;
        t = h * (HB * (HB + 1) / 2) + P * HB - P * (P - 1) / 2 + (Q - P);
    } else {
        t = P * NB - P * (P - 1) / 2 + (Q - P);
    }
    return D[t * 64 + (lo & 7) * 8 + (hi & 7)];
}

// Entry (p, q), p <= q, of the packed upper triangle of G (v = (A, B, J_0.., N_0..), include/varsens_b200.h) from the combined CTA sums.
// Paired layout (Grams of w = (P, A, B) and u = (M, A, B), HS coordinates each): first-order entries are exact recombinations
// (A.J_j = (A.P_j - A.M_j)/2, A.N_j = (A.P_j + A.M_j)/2); the J/N blocks come out symmetrised,
//   G[J_i][J_j] = G[N_i][N_j] = (N_i.N_j + J_i.J_j)/2,   G[J_i][N_j] = (N_i.J_j + J_i.N_j)/2,
// which is all the estimators read (they add the two members of each pair, saltelli.py:612-613,618-619).
template <int K, int NB, int HB, bool PM>
__device__ __forceinline__ double packed_pq(const double *__restrict__ D, int p, int q) {      // p <= q
    if constexpr (!PM) {
        return dense_at<NB, HB, PM>(D, p, q);
    } else {
        constexpr int HS = 8 * HB;
        auto Dd = [&](int x, int y) { return dense_at<NB, HB, PM>(D, x, y); };
        if (q < 2) return Dd(K + p, K + q);                           // A.A, A.B, B.B (w triangle)
        if (p < 2) {
            const bool qn = q >= 2 + K;
            const int j = qn ? q - 2 - K : q - 2;
            const double ap = Dd(j, K + p), am = Dd(HS + j, HS + K + p);
            return 0.5 * (qn ? ap + am : ap - am);
        }
        const bool pn = p >= 2 + K, qn = q >= 2 + K;
        const int i = pn ? p - 2 - K : p - 2, j = qn ? q - 2 - K : q - 2;
        const double pp = Dd(i, j), mm = Dd(HS + i, HS + j);
        return 0.25 * (pn == qn ? pp + mm : pp - mm);
    }
}

template <int K, int NB, int HB, bool PM>
__host__ __device__ constexpr size_t wsd_tail_smem_doubles() {
    constexpr int LROW = wsd_lrow<NB, HB, PM>();
    constexpr int m = 2 + 2 * K, plen = 4 + m * (m + 1) / 2, rlen = (int)result_len(K, 1);
    return (size_t)128 + LROW + 2 * (size_t)(plen + 4) + rlen + 8;      // combine scratch | D | Pk | Pr | R
}

// Sum of `nrows` rows (LROW doubles each, row r at rows[r * LROW]) in row order into D (shared).  One double2 column (= one lane's
// C fragment of one tile) per thread with 16 independent loads in flight; the four shifted sums by warp 0, lane l adding rows
// l, l+32, ... in order and then the lanes in lane order.  Fixed order -> bit-reproducible.  All threads of the CTA call it.
template <int NTL, int LROW>
__device__ __forceinline__ void combine_rows(const double *__restrict__ rows, int nrows, double *__restrict__ D, double *__restrict__ ps) {
    constexpr int L2 = LROW / 2;
    const int tid = threadIdx.x, nthr = blockDim.x;
    const double2 *base = reinterpret_cast<const double2 *>(rows);
    for (int c2 = tid; c2 < NTL * 32; c2 += nthr) {
        const double2 *src = base + c2;
        double2 acc = make_double2(0.0, 0.0);
        for (int b = 0; b < nrows; b += 16) {           // 16 independent loads in flight, predicated (a short tail is one round trip too)
            double2 v[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) v[u] = (b + u < nrows) ? __ldcg(src + (size_t)(b + u) * L2) : make_double2(0.0, 0.0);
#pragma unroll
            for (int u = 0; u < 16; ++u) { acc.x += v[u].x; acc.y += v[u].y; }
        }
        reinterpret_cast<double2 *>(D)[c2] = acc;
    }
    if (tid < 32) {
        double2 s01 = make_double2(0.0, 0.0), s23 = make_double2(0.0, 0.0);
        for (int b = tid; b < nrows; b += 32) {
            const double2 v0 = __ldcg(base + (size_t)b * L2 + NTL * 32), v1 = __ldcg(base + (size_t)b * L2 + NTL * 32 + 1);
            s01.x += v0.x; s01.y += v0.y; s23.x += v1.x; s23.y += v1.y;
        }
        double *lane4 = ps + tid * 4;
        lane4[0] = s01.x; lane4[1] = s01.y; lane4[2] = s23.x; lane4[3] = s23.y;
        __syncwarp();
        if (tid < 8) {
            double v = 0.0;
            if (tid < 4)
                for (int l = 0; l < 32; ++l) v += ps[l * 4 + tid];
            D[NTL * 64 + tid] = v;
        }
    }
    __syncthreads();
}

// varsens/saltelli.py:577-622 for a scalar objective and compile-time K: finalize_body (device.cuh) with every index
// computation folded at compile time (the generic form spends most of its ~6 us on run-time integer divisions).  Same
// operations in the same order on the same operands, hence the same bits.  R = E_2 var_y U_j U_nj sens sens_t sens_2 sens_2n.
template <int K>
__device__ __forceinline__ void finalize_fixed(double n, double rows, const double *__restrict__ P, double *__restrict__ R) {
    constexpr int m = 2 + 2 * K;
    const double *G = P + 4;
    auto at = [&](int p, int q) { return G[p * m - p * (p - 1) / 2 + (q - p)]; };           // p <= q
    auto sym = [&](int p, int q) { return p <= q ? at(p, q) : at(q, p); };
    const double e2 = at(0, 1) / n;                                                           // :577
    const double tot = P[0] + P[1];
    const double var = (P[2] + P[3] - tot * tot / (2.0 * rows)) / (2.0 * rows - 1.0);         // :583
    double *Uj = R + 2, *Unj = Uj + K, *sens = Unj + K, *senst = sens + K, *s2 = senst + K, *s2n = s2 + K * K;
    const int tid = threadIdx.x, nthr = blockDim.x;
    if (tid == 0) { R[0] = e2; R[1] = var; }
    for (int j = tid; j < K; j += nthr) {
        const int iJ = 2 + j, iN = 2 + K + j;
        double uj = at(0, iJ) / (n - 1.0);                                                    // :591-593
        uj += at(1, iN) / (n - 1.0);
        uj /= 2.0;
        double unj = at(0, iN) / (n - 1.0);                                                   // :594-596
        unj += at(1, iJ) / (n - 1.0);
        unj /= 2.0;
        Uj[j] = uj;
        Unj[j] = unj;
        sens[j] = (uj - e2) / var;                                                            // :608
        senst[j] = 1.0 - ((unj - e2) / var);                                                  // :609
    }
    for (int e = tid; e < K * K; e += nthr) {
        const int i = e / K, j = e - i * K;
        const int Ji = 2 + i, Ni = 2 + K + i, Jj = 2 + j, Nj = 2 + K + j;
        double v2 = at(Jj < Ni ? Jj : Ni, Jj < Ni ? Ni : Jj) + at(Ji < Nj ? Ji : Nj, Ji < Nj ? Nj : Ji);     // :612-613 (J < N always)
        v2 /= 2.0 * (n - 1.0);
        v2 -= e2;
        v2 /= var;
        double v2n = sym(Ni, Nj) + sym(Ji, Jj);                                               // :618-619
        v2n /= 2.0 * (n - 1.0);
        v2n -= e2;
        v2n /= var;
        s2[e] = v2;
        s2n[e] = v2n;
    }
}

// Runs in the CTA that completes the second-level combine (all threads).  On entry D (shared) holds the sums over all CTAs.
template <int K, int NB, int HB, bool PM>
__device__ __forceinline__ void fused_tail(const FusedTail &tail, double *__restrict__ smem, unsigned long long t0, unsigned long long ta,
                                           unsigned long long tb, unsigned long long tc) {
    constexpr int LROW = wsd_lrow<NB, HB, PM>();
    constexpr int NTL = wsd_ntl<NB, HB, PM>();
    constexpr int m = 2 + 2 * K, plen = 4 + m * (m + 1) / 2, rlen = (int)result_len(K, 1);
    double *D = smem + 128;                                // [LROW] (after the combine scratch)
    double *Pk = D + LROW;                                 // [plen] packed partial sums of this rank
    double *Pr = Pk + plen + 4;                            // [plen] reduced over ranks (mode 2)
    double *R = Pr + plen + 4;                             // [rlen] results
    const int tid = threadIdx.x, nthr = blockDim.x;
    // packed partial-sum vector: warp w takes rows p = w, w + nwarp, ... of the upper triangle, lanes run over q >= p
    if (tid < 4) {
        Pk[tid] = D[NTL * 64 + tid];
        if (tail.partials) tail.partials[tid] = Pk[tid];
    }
    for (int p = tid >> 5; p < m; p += nthr >> 5) {
        const int row0 = 4 + p * m - p * (p - 1) / 2 - p;                    // index of (p, q) is row0 + q
        for (int q = p + (tid & 31); q < m; q += 32) {
            const double v = packed_pq<K, NB, HB, PM>(D, p, q);
            Pk[row0 + q] = v;
            if (tail.partials) tail.partials[row0 + q] = v;
        }
    }
    __syncthreads();
    if (tail.mode == 0) return;
    const unsigned long long t1 = globaltimer_ns();
    unsigned long long t2 = t1, t3 = t1;
    const double *Pfin = Pk;
    __shared__ unsigned timed_out;
    if (tid == 0) timed_out = 0u;
    __syncthreads();
    if (tail.mode == 2) {
        // all-reduce over NVLink peer memory, low-latency protocol (device.cuh: ll_push / ll_reduce): one warp per peer
        // stores my vector as 16-byte {lo, epoch, hi, epoch} units into slot `rank` of every rank's buffer; then every
        // thread polls the tags of "its" elements in my own buffer and adds the world slots in rank order.
        ll_push(tail.peer_bufs, tail.world, tail.rank, tail.epoch, plen, Pk);
        t2 = globaltimer_ns();
        if (!ll_reduce(tail.peer_bufs, tail.world, tail.rank, tail.epoch, plen, Pr, tail.timeout_ns)) timed_out = 1u;
        __syncthreads();
        t3 = globaltimer_ns();
        Pfin = Pr;
    }
    // estimators
    finalize_fixed<K>(tail.n_total, tail.rows_total, Pfin, R);
    __syncthreads();
    for (int e = tid; e < rlen; e += nthr) {
        const double v = R[e];
        if (tail.res_dev) tail.res_dev[e] = v;
        if (tail.res_host) tail.res_host[e] = v;
    }
    if (tail.res_host && tid == 0) {
        tail.res_host[rlen + HOST_RES_STATUS] = timed_out ? 1.0 : 0.0;
        double *x = tail.res_host + rlen + HOST_RES_STAMPS;
        x[0] = (double)(t1 - t0);                       // two-level combine (this CTA's share) + pack, ns
        x[1] = (double)(t2 - t1);                       // peer stores (issue)
        x[2] = (double)(t3 - t2);                       // wait for the peers' elements + rank-order sum
        x[3] = (double)(globaltimer_ns() - t3);         // estimators + result stores
        x[4] = (double)(ta - t0);                       // first-level combine (my group's rows)
        x[5] = (double)(tb - ta);                       // group row to HBM + fence + second-level ticket
        x[6] = (double)(tc - tb);                       // second-level combine
        x[7] = (double)(t1 - tc);                       // packed partial-sum vector
    }
}

// Coordinate d (run-time: lane = coordinate, no divergence) of the Halton point m from the fixed-layout shared table; used
// once per CTA, for the common shift.  Bases and row offsets come from a compile-time table.
template <int K>
struct FixedTab {
    uint32_t base[K], off[K];
};
template <int K>
__host__ __device__ constexpr FixedTab<K> make_fixed_tab() {
    FixedTab<K> t{};
    for (int d = 0; d < K; ++d) {
        t.base[d] = prime_at(d);
        t.off[d] = d == 0 ? 0u : foff(d);
    }
    return t;
}
template <int K>
__device__ __forceinline__ double halton_coord_fixed(const double *__restrict__ terms, int d, uint32_t m) {
    constexpr FixedTab<K> tab = make_fixed_tab<K>();
    if (d == 0) return (double)__brev(m) * 2.3283064365386962890625e-10;
    const uint32_t b = tab.base[d];
    const double *row = terms + tab.off[d];
    double x = 0.0;
    while (m != 0u) {
        const uint32_t q = m / b;
        x = __dadd_rn(x, row[m - q * b]);
        row += b;
        m = q;
    }
    return x;
}

template <int K, class F, bool SEPARABLE, int EPS, int NBUF, int IB>
__global__ void __launch_bounds__((EPS + 1) * WS_S * 32, 1)
fused_wsd_kernel(SourceDev src, FusedConst<K> fc, F f, uint64_t i_begin, uint64_t i_end, FusedTail tail) {
    constexpr int WS_E = EPS * WS_S;
    constexpr int M = 2 + 2 * K;
    constexpr bool PM = wsd_paired<K, F, SEPARABLE>();  // paired tile layout (see pm_pays)
    constexpr int HB = pm_hb<K>();
    constexpr int NB = PM ? 2 * HB : (M + 7) / 8;       // 8-wide blocks of a tile row
    constexpr int MPAD = NB * 8;
    constexpr int NTL = wsd_ntl<NB, HB, PM>();          // 8x8 tiles: two upper triangles / one
    constexpr int LROW = wsd_lrow<NB, HB, PM>();
    constexpr int TILE = MPAD * YT_PITCH;               // doubles per Y tile

    extern __shared__ double smem[];
    __shared__ double xs_sh[K];
    __shared__ double shift_sh;
    __shared__ unsigned last_sh;
    const unsigned long long t_entry = globaltimer_ns();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t nterms = src.raw ? 0u : ((foff(K) + 1u) & ~1u);     // even: the table is copied 16 bytes at a time
    double *terms = smem;
    volatile double *tokp = smem + nterms;                                    // opaque functor token (see the functors)
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + nterms + 1);        // full[WS_E][NBUF], empty[WS_E][NBUF]
    double *tiles = smem + nterms + 1 + 2 * NBUF * WS_E;                      // [WS_E][NBUF][TILE]
    if (nterms) load_fixed_table<K>(terms, src.h, fc);
    for (int e = threadIdx.x; e < WS_E * NBUF * TILE; e += blockDim.x) tiles[e] = 0.0;
    if (threadIdx.x == 0) {
        *tokp = F::token;
        for (int b = 0; b < 2 * NBUF * WS_E; ++b) mbar_init(bars + b, 1);
    }
    __syncthreads();
    // common shift of the variance sums, f(M_1[0]): every CTA (and every rank) derives the same bits from base row 0
    if (threadIdx.x < K) {                                // lane = coordinate: the table reads of the K chains overlap
        const int d = threadIdx.x;
        double p = src.raw ? src.raw[d] : halton_coord_fixed<K>(terms, d, (uint32_t)src.start);
        if (fc.scale_kind == VS_SCALE_LINEAR) p = scale_value(VS_SCALE_LINEAR, fc.lb[d], fc.wr[d], p);
        else if (fc.scale_kind == VS_SCALE_POWER) p = scale_value(VS_SCALE_POWER, fc.lb[d], fc.wr[d], p);
        xs_sh[d] = p;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double x[K];
#pragma unroll
        for (int c = 0; c < K; ++c) x[c] = xs_sh[c];
        shift_sh = f(x, F::token);
    }
    __syncthreads();
    auto full_bar = [&](int e, int slot) { return bars + (e * NBUF + slot); };
    auto empty_bar = [&](int e, int slot) { return bars + NBUF * WS_E + (e * NBUF + slot); };
    const unsigned long long t_pro = globaltimer_ns();

    const uint64_t rows = i_end - i_begin;
    const uint64_t nbatch = (rows + 31) / 32;
    const uint64_t G = (uint64_t)gridDim.x * WS_E;
    // E-warp e of this CTA takes batches first_batch(e), + G, + 2G, ...  The order is team-major (team = e / WS_S: every
    // sub-partition has one E-warp of each team), so the warps that get one batch more than the others when nbatch is not a
    // multiple of G are spread one per sub-partition: their last batch then runs alone on its FP64 pipe (~5.5 us) instead of
    // sharing it with a second straggler (~10.8 us) -- at 8 GPUs (55.35 batches per warp) that is ~1 % of the step.
    auto first_batch = [&](int e) -> uint64_t {
        return (uint64_t)(e / WS_S) * ((uint64_t)gridDim.x * WS_S) + (uint64_t)blockIdx.x * WS_S + (uint64_t)(e % WS_S);
    };
    auto count_of = [&](int e) -> uint64_t {
        const uint64_t g = first_batch(e);
        return g < nbatch ? (nbatch - g + G - 1) / G : 0;
    };
    double sA = 0.0, qA = 0.0, sB = 0.0, qB = 0.0;
    double acc[NTL][2];
#pragma unroll
    for (int t = 0; t < NTL; ++t) { acc[t][0] = 0.0; acc[t][1] = 0.0; }

    if (warp >= WS_S) {
        // ------------------------------------ E-warp ------------------------------------
        const int e = warp - WS_S;
        const double shift = shift_sh;
        const uint64_t basehi = table_basehi(terms);
        const uint64_t cnt = count_of(e);
        uint64_t bt = first_batch(e);
        for (uint64_t it = 0; it < cnt; ++it, bt += G) {
            const int slot = (int)(it % NBUF);
            double a[K], b[K];
            const bool tr_on = fc.trace && blockIdx.x == 0 && lane == 0 && it < 64;
            long long *trp = fc.trace + ((size_t)warp * 64 + (it < 64 ? it : 0)) * 4;
            if (tr_on) trp[0] = clock64();
            const bool valid = gen_rows<K, IB>(src, fc, basehi, i_begin, rows, bt, lane, [&](int d, double xa, double xb) {
                a[d] = xa;
                b[d] = xb;
            });
            if (tr_on) trp[1] = clock64();
            mbar_wait(empty_bar(e, slot), (uint32_t)(((it / NBUF) & 1) ^ 1), MBAR_HINT_NS);
            if (tr_on) trp[2] = clock64();
            double *Y = tiles + ((size_t)e * NBUF + slot) * TILE;
            eval_rows<K, F, SEPARABLE, PM>(f, tokp, a, b, valid, Y + lane, shift, sA, qA, sB, qB, YT_PITCH);
            __syncwarp();
            if (tr_on) trp[3] = clock64();
            if (lane == 0) mbar_arrive(full_bar(e, slot));
        }
    } else {
        // ------------------------------------ S-warp ------------------------------------
        uint64_t cn[EPS], cmax = 0;
#pragma unroll
        for (int h = 0; h < EPS; ++h) {
            cn[h] = count_of(warp + h * WS_S);
            cmax = cn[h] > cmax ? cn[h] : cmax;
        }
        const int foff = (lane >> 2) * YT_PITCH + (lane & 3);   // fragment element of this lane inside an 8-row block
        for (uint64_t it = 0; it < cmax; ++it) {
            const int slot = (int)(it % NBUF);
            const uint32_t par = (uint32_t)((it / NBUF) & 1);
#pragma unroll
            for (int h = 0; h < EPS; ++h) {
                const int e = warp + h * WS_S;
                if (it >= cn[h]) continue;
                const bool tr_on = fc.trace && blockIdx.x == 0 && lane == 0 && it < 32;
                long long *trp = fc.trace + ((size_t)warp * 64 + (it < 32 ? it * EPS + h : 0)) * 4;
                if (tr_on) trp[0] = clock64();
                mbar_wait(full_bar(e, slot), par, MBAR_HINT_NS);
                if (tr_on) trp[1] = clock64();
                const double *Y = tiles + ((size_t)e * NBUF + slot) * TILE + foff;
#pragma unroll 2
                for (int r0 = 0; r0 < 32; r0 += 4) {
                    double fr[NB];
#pragma unroll
                    for (int P = 0; P < NB; ++P) fr[P] = Y[P * 8 * YT_PITCH + r0];
                    for_each_tile<NB, HB, PM>([&](int t, int P, int Q) { dmma_m8n8k4(acc[t][0], acc[t][1], fr[P], fr[Q]); });
                }
                __syncwarp();
                if (tr_on) trp[2] = clock64();
                if (lane == 0) mbar_arrive(empty_bar(e, slot));
            }
        }
    }

    // ---- combine: every S-warp drops its C fragments into a compact tile-major image, summed in S-warp order ----
    __syncthreads();
    const unsigned long long t_loop = globaltimer_ns();
    double *img = smem;                                   // [WS_S][NTL*64] then [WS_E][4]
    double *sums = img + (size_t)WS_S * NTL * 64;
    if (warp < WS_S) {
        double2 *mine = reinterpret_cast<double2 *>(img + (size_t)warp * NTL * 64);
#pragma unroll
        for (int t = 0; t < NTL; ++t) mine[t * 32 + lane] = make_double2(acc[t][0], acc[t][1]);
    } else {
        sA = warp_sum(sA); qA = warp_sum(qA); sB = warp_sum(sB); qB = warp_sum(qB);
        if (lane == 0) {
            double *s4 = sums + (warp - WS_S) * 4;
            s4[0] = sA; s4[1] = sB; s4[2] = qA; s4[3] = qB;
        }
    }
    __syncthreads();
    double *bp = tail.blockpart + (size_t)blockIdx.x * LROW;
    for (int e = threadIdx.x; e < NTL * 64; e += blockDim.x) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < WS_S; ++w) v += img[(size_t)w * NTL * 64 + e];
        bp[e] = v;
    }
    if (threadIdx.x < 8) {
        double v = 0.0;
        if (threadIdx.x < 4)
            for (int w = 0; w < WS_E; ++w) v += sums[w * 4 + threadIdx.x];
        bp[NTL * 64 + threadIdx.x] = v;
    }
    // ---- two-level ticket.  The last CTA of each group of TAIL_GROUP consecutive CTAs sums its group's rows (in CTA order); the
    //      last group to finish sums the group rows (in group order) and runs the tail.  Which CTA does the work depends on
    //      timing, what it computes does not.  One SM pulling all 148 rows (0.9 MB) through its L2 port took ~10 us; a group
    //      of 16 rows plus 10 group rows take ~2. ----
    const int group = blockIdx.x / TAIL_GROUP, ngroups = (gridDim.x + TAIL_GROUP - 1) / TAIL_GROUP;
    const int gfirst = group * TAIL_GROUP;
    const int gsize = (gfirst + TAIL_GROUP <= (int)gridDim.x) ? TAIL_GROUP : (int)gridDim.x - gfirst;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned t = atomicAdd(tail.ticket + 1 + group, 1u);
        last_sh = (t == (unsigned)gsize - 1u) ? 1u : 0u;
        if (last_sh) tail.ticket[1 + group] = 0u;
    }
    __syncthreads();
    if (!last_sh) return;
    __threadfence();
    const unsigned long long t0 = globaltimer_ns();
    double *ps = smem, *D = smem + 128;
    combine_rows<NTL, LROW>(tail.blockpart + (size_t)gfirst * LROW, gsize, D, ps);
    const unsigned long long ta = globaltimer_ns();
    unsigned long long tb = ta, tc = ta;
    if (ngroups > 1) {
        double *gp = tail.grouppart + (size_t)group * LROW;
        for (int e = threadIdx.x; e < LROW; e += blockDim.x) gp[e] = D[e];
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) {
            const unsigned t = atomicAdd(tail.ticket, 1u);
            last_sh = (t == (unsigned)ngroups - 1u) ? 1u : 0u;
            if (last_sh) tail.ticket[0] = 0u;
        }
        __syncthreads();
        if (!last_sh) return;
        __threadfence();
        tb = globaltimer_ns();
        combine_rows<NTL, LROW>(tail.grouppart, ngroups, D, ps);
        tc = globaltimer_ns();
    }
    fused_tail<K, NB, HB, PM>(tail, smem, t0, ta, tb, tc);
    if (tail.mode >= 1 && tail.res_host && threadIdx.x == 0) {      // this CTA's own phases (diagnostics)
        double *x = tail.res_host + result_len(K, 1) + HOST_RES_STAMPS;
        x[8] = (double)(t_pro - t_entry);                            // prologue: table copy, tile zeroing, barriers, shift
        x[9] = (double)(t_loop - t_pro);                             // main loop
        x[10] = (double)(t0 - t_loop);                               // CTA combine + row to HBM + fence + first-level ticket
    }
}

// f(M_1[0]): the common shift for the variance sums (identical on every rank) -- separate launch, used by the single-role
// fused_kernel only (the warp-specialised kernel computes it in its prologue).
template <int K, class F>
__global__ void shift_kernel(SourceDev src, FusedConst<K> fc, F f, double *out) {
    __shared__ double xs[K];
    const int d = threadIdx.x;                     // one thread per coordinate: the table reads of the K chains overlap
    if (d < K) {
        double p = src.raw ? src.raw[d] : halton_coord(src.h, d, (uint32_t)src.start);
        if (fc.scale_kind == VS_SCALE_LINEAR) p = scale_value(VS_SCALE_LINEAR, fc.lb[d], fc.wr[d], p);
        else if (fc.scale_kind == VS_SCALE_POWER) p = scale_value(VS_SCALE_POWER, fc.lb[d], fc.wr[d], p);
        xs[d] = p;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double x[K];
#pragma unroll
        for (int c = 0; c < K; ++c) x[c] = xs[c];
        *out = f(x, F::token);
    }
}

// kernel variant (VS_FUSED_VARIANT overrides; see DESIGN.md "fused kernel variants"):
//   1 = single-role warps, register-tile Gram (also the first-order-only kernel; separate shift / scatter launches)
//   5 = E/S warp-specialised, 2 E-warps per S-warp, DMMA Gram   6 = same with 3 E-warps per S-warp     (one launch per step)
// default: 6 (k <= 18: 1-13 % faster than 5, tools/variant_sweep.py).  At k >= 20 the 12-warp form (168 registers per thread, no
// spills) was the faster one while generation was table-bound (n = 2^24: 4.79 vs 5.06 ms); since the PTX digit step and the
// computed terms it is the other way round for the generic functor on ONE GPU -- k = 20, n = 2^24: 4.45 vs 4.51 ms per step,
// same-box A/B.  It is also the less even one: its slowest CTA finishes 15-60 us after the others (12 E-warps share the batches
// of a CTA less evenly than 8) and its kernel time jitters by 0.5 % against 0.02 %, which the peer-memory step of a multi-GPU
// run pays as waiting for the slowest rank: 8 GPUs 0.647 vs 0.635 ms per step, e2e 0.737 vs 0.707.  So: 6 for single-GPU steps
// of at least 2^22 rows with the generic functor; 5 for peer-exchange steps, small shards and the separable shortcut (3.02 vs
// 3.21 ms).
template <int K>
static int fused_variant_for(const vs_ctx *c, bool second, bool separable, uint64_t rows, bool peer) {
    if (!second) return 1;
    const int v = c->opt.fused_variant;
    if (v == 1 || v == 5 || v == 6) return v;
    if (K < 20) return 6;
    return (!separable && !peer && rows >= (1ull << 22)) ? 6 : 5;
}

template <int K, class F, bool SECOND, bool SEPARABLE>
static int launch_fused_t(vs_ctx *c, const SourceDev &src, const FusedConst<K> &fc, const F &f, uint64_t i_begin, uint64_t i_end,
                          double *partials, const FusedReq *req, bool *finalized) {
    constexpr int M = 2 + 2 * K;
    constexpr int T = SECOND ? gram_tile_for(M) : 2;
    constexpr int NT = (M + T - 1) / T;
    constexpr int MP = (NT * T) % 2 ? NT * T : NT * T + 1;
    constexpr int NTILES = SECOND ? NT * (NT + 1) / 2 : NT;
    constexpr int TPL = SECOND ? 1 : (NTILES + 31) / 32;
    constexpr int PER_BLOCK = TPL * 32 * T * T + 4;
    const uint32_t nterms = src.raw ? 0u : ((foff(K) + 1u) & ~1u);     // even: the table is copied 16 bytes at a time
    const uint64_t rows = i_end - i_begin;
    const uint64_t nbatch = (rows + 31) / 32;
    const int variant = fused_variant_for<K>(c, SECOND, SEPARABLE, rows, req && req->mode == 2);
    *finalized = false;
    if constexpr (SECOND) {
        if (variant == 5 || variant == 6) {
            constexpr bool PMk = wsd_paired<K, F, SEPARABLE>();
            constexpr int HBk = pm_hb<K>();
            constexpr int NBk = PMk ? 2 * HBk : (M + 7) / 8, MPADk = NBk * 8;
            constexpr int LROWk = wsd_lrow<NBk, HBk, PMk>(), NTLk = wsd_ntl<NBk, HBk, PMk>();
            const int eps = variant == 6 ? 3 : 2;
            uint64_t wantd = (nbatch + eps * WS_S - 1) / (eps * WS_S);
            int gridd = (int)(wantd < (uint64_t)c->sm_count ? wantd : (uint64_t)c->sm_count);
            if (gridd < 1) gridd = 1;
            const int ngroups = (gridd + TAIL_GROUP - 1) / TAIL_GROUP;
            VS_REQUIRE(ngroups < 60, VS_ERR_UNSUPPORTED, "grid of %d CTAs needs more ticket counters than the ctx holds", gridd);
            VS_TRY(ensure(c, c->block_buf, (size_t)(gridd + ngroups) * LROWk * sizeof(double)));
            if (!c->ticket_buf.p) {
                VS_TRY(ensure(c, c->ticket_buf, 256));
                VS_CUDA(cudaMemsetAsync(c->ticket_buf.p, 0, 256, c->stream));
            }
            FusedTail tail{};
            tail.blockpart = (double *)c->block_buf.p;
            tail.grouppart = (double *)c->block_buf.p + (size_t)gridd * LROWk;
            tail.poll_perm = (req && req->poll_perm) ? 1 : 0;
            tail.ticket = (unsigned *)c->ticket_buf.p;
            tail.partials = partials;
            tail.mode = req ? req->mode : 0;
            if (tail.mode >= 1) {
                VS_TRY(ensure_host_res(c, result_len(K, 1) + HOST_RES_EXTRA));
                tail.res_dev = nullptr;                              // results go straight to mapped host memory
                tail.res_host = c->host_res;
                tail.n_total = (double)req->n_total;
                tail.rows_total = (double)req->rows_total;
                tail.world = req->world;
                tail.rank = req->rank;
                tail.epoch = req->epoch;
                tail.peer_bufs = req->peer_bufs_dev;
                tail.peer_flags = req->peer_flags_dev;
                tail.timeout_ns = (unsigned long long)c->opt.p2p_timeout_ms * 1000000ull;
            }
            size_t smem_run = ((size_t)nterms + 1 + 2 * eps * WS_S + (size_t)eps * WS_S * MPADk * YT_PITCH) * sizeof(double);
            size_t smem_red = ((size_t)WS_S * NTLk * 64 + 4 * eps * WS_S) * sizeof(double);
            size_t smem_tail = wsd_tail_smem_doubles<K, NBk, HBk, PMk>() * sizeof(double);
            size_t smem = smem_run > smem_red ? smem_run : smem_red;
            if (smem_tail > smem) smem = smem_tail;
            VS_REQUIRE(smem <= c->smem_optin, VS_ERR_UNSUPPORTED, "fused kernel needs %zu bytes of shared memory", smem);
            // index-bit class: runs whose Halton indices all stay below 2^26 (every BASELINE config) visit fewer digit positions
            const bool ib26 = !src.raw && (src.start + 2 * src.n - 1) < (1ull << 26) && c->opt.index_bits != 32;
#ifdef VS_EXP_MINIMAL                                            // experiment builds: one instantiation only
            VS_REQUIRE(ib26 && variant == 5, VS_ERR_UNSUPPORTED, "experiment build: variant 5, indices < 2^26 only");
            auto kern = fused_wsd_kernel<K, F, SEPARABLE, 2, 1, 26>;
#else
            auto kern = variant == 6 ? (ib26 ? fused_wsd_kernel<K, F, SEPARABLE, 3, 1, 26> : fused_wsd_kernel<K, F, SEPARABLE, 3, 1, 32>)
                                     : (ib26 ? fused_wsd_kernel<K, F, SEPARABLE, 2, 1, 26> : fused_wsd_kernel<K, F, SEPARABLE, 2, 1, 32>);
#endif
            const int ki = (variant == 6 ? 2 : 0) + (ib26 ? 1 : 0);
            static size_t smem_set[64][4] = {};                  // per instantiation and device: set the attribute once per size
            if (c->device >= 64 || smem_set[c->device][ki] < smem) {
                VS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                if (c->device < 64) smem_set[c->device][ki] = smem;
            }
            time_begin(c);
            FusedConst<K> fcl = fc;
            fcl.poll_perm = tail.poll_perm;
            kern<<<gridd, (eps + 1) * WS_S * 32, smem, c->stream>>>(src, fcl, f, i_begin, i_end, tail);
            time_end(c);
            c->launches++;
            VS_CUDA(cudaGetLastError());
            *finalized = tail.mode >= 1;
            if (fc.trace) {                                  // profiling only: dump CTA 0's clock stamps
                std::vector<long long> h(16 * 64 * 4);
                VS_CUDA(cudaMemcpyAsync(h.data(), fc.trace, h.size() * sizeof(long long), cudaMemcpyDeviceToHost, c->stream));
                VS_CUDA(cudaStreamSynchronize(c->stream));
                if (FILE *fp = fopen(c->opt.trace.c_str(), "w")) {
                    for (int w = 0; w < 16; ++w)
                        for (int i = 0; i < 64; ++i) {
                            const long long *r = &h[((size_t)w * 64 + i) * 4];
                            if (r[0]) fprintf(fp, "%d %d %lld %lld %lld %lld\n", w, i, r[0], r[1], r[2], r[3]);
                        }
                    fclose(fp);
                }
            }
            return VS_OK;
        }
    }
    VS_REQUIRE(partials, VS_ERR_ARG, "this fused kernel variant needs a partial-sum buffer");
    VS_REQUIRE(!(req && req->poll_perm), VS_ERR_UNSUPPORTED, "this fused kernel variant cannot poll a permutation in flight");
    const int ewarps = FUSED_WARPS;
    uint64_t want = (nbatch + ewarps - 1) / ewarps;
    int grid = (int)(want < (uint64_t)c->sm_count ? want : (uint64_t)c->sm_count);
    if (grid < 1) grid = 1;
    VS_TRY(ensure(c, c->block_buf, (size_t)grid * PER_BLOCK * sizeof(double)));
    VS_TRY(ensure(c, c->misc_buf, 64));
    shift_kernel<K, F><<<1, (K + 31) / 32 * 32, 0, c->stream>>>(src, fc, f, (double *)c->misc_buf.p);
    c->launches++;
    {
        size_t smem_run = ((size_t)nterms + 1 + (size_t)FUSED_WARPS * 32 * MP) * sizeof(double);
        size_t smem_red = ((size_t)TPL * 32 * T * T + 4) * sizeof(double);
        size_t smem = smem_run > smem_red ? smem_run : smem_red;
        VS_REQUIRE(smem <= c->smem_optin, VS_ERR_UNSUPPORTED, "fused kernel needs %zu bytes of shared memory", smem);
        auto kern = fused_kernel<K, F, SECOND, SEPARABLE>;
        VS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        time_begin(c);
        kern<<<grid, FUSED_WARPS * 32, smem, c->stream>>>(src, fc, f, i_begin, i_end, (const double *)c->misc_buf.p,
                                                          (double *)c->block_buf.p);
        time_end(c);
    }
    c->launches++;
    VS_CUDA(cudaGetLastError());
    GramGeom g{};
    g.m = M; g.l = 1; g.T = T; g.nt = NT; g.mp = MP;
    g.tr_max = SECOND ? NT : 1;
    g.ntiles = NTILES; g.LG = 32; g.RG = 1; g.R = 32; g.passes = TPL;
    return launch_gram_scatter(c, g, grid, (const double *)c->block_buf.p, partials, (int)vs_partials_len(K, 1));
}

template <int K>
static int fill_const(vs_ctx *c, const SourceDev &src, const ScaleDev &s, FusedConst<K> &fc) {
    fc.scale_kind = s.kind;
    const double *h = s.host;                                   // lb | wr
    for (int d = 0; d < K; ++d) {
        fc.lb[d] = s.kind != VS_SCALE_IDENTITY ? h[d] : 0.0;
        fc.wr[d] = s.kind != VS_SCALE_IDENTITY ? h[K + d] : 1.0;
    }
    fc.small_index = 0;
    fc.poll_perm = 0;
    fc.trace = nullptr;
    for (int u = 0; u < FusedConst<K>::AR_N; ++u)
        for (int j = 0; j < HL_J; ++j) { fc.arh[u][j] = 0.0; fc.arl[u][j] = 0.0; }
    if (!c->opt.trace.empty()) {
        VS_TRY(ensure(c, c->dir_buf, 16 * 64 * 4 * sizeof(long long)));
        VS_CUDA(cudaMemsetAsync(c->dir_buf.p, 0, 16 * 64 * 4 * sizeof(long long), c->stream));
        fc.trace = (long long *)c->dir_buf.p;
    }
    if (!src.raw) {
        fc.small_index = (src.start + 2 * src.n - 1) < (1ull << 29) ? 1 : 0;
        if (K > AR_D0) {
            VS_REQUIRE(c->halton.arith_ok, VS_ERR_UNSUPPORTED, "computed Halton terms do not reproduce the term table in mode %d",
                       c->halton.mode);
            for (int u = 0; u < K - AR_D0; ++u)
                for (int j = 0; j < HL_J; ++j) {
                    fc.arh[u][j] = c->halton.arh[(size_t)(AR_D0 + u) * HL_J + j];
                    fc.arl[u][j] = c->halton.arl[(size_t)(AR_D0 + u) * HL_J + j];
                }
        }
        VS_REQUIRE(src.h.fixed && src.h.fixed_len >= foff(K), VS_ERR_ARG, "fixed-layout Halton table missing (%u of %u doubles)",
                   src.h.fixed_len, (uint32_t)foff(K));
    }
    return VS_OK;
}

template <int K>
static int dispatch_k(vs_ctx *c, const SourceDev &src, const ScaleDev &s, const ObjectiveDev &o, uint64_t i_begin, uint64_t i_end,
                      int flags, double *partials, const FusedReq *req, bool *finalized) {
    FusedConst<K> fc;
    VS_TRY(fill_const<K>(c, src, s, fc));
    const bool second = flags & VS_FLAG_SECOND_ORDER, sep = flags & VS_FLAG_SEPARABLE;
    const double *hp = o.host;
    if (o.id == VS_OBJ_GFUNCTION) {
        GFunctionReg<K> f;
        f.C = 1.0;
        for (int d = 0; d < K; ++d) { f.a[d] = hp[d]; f.C *= hp[K + d]; }
#ifdef VS_EXP_MINIMAL
        VS_REQUIRE(second && !sep, VS_ERR_UNSUPPORTED, "experiment build: generic second-order kernel only");
        return launch_fused_t<K, GFunctionReg<K>, true, false>(c, src, fc, f, i_begin, i_end, partials, req, finalized);
#else
        if (second) {
            if (sep) return launch_fused_t<K, GFunctionReg<K>, true, true>(c, src, fc, f, i_begin, i_end, partials, req, finalized);
            return launch_fused_t<K, GFunctionReg<K>, true, false>(c, src, fc, f, i_begin, i_end, partials, req, finalized);
        }
        if (sep) return launch_fused_t<K, GFunctionReg<K>, false, true>(c, src, fc, f, i_begin, i_end, partials, req, finalized);
        return launch_fused_t<K, GFunctionReg<K>, false, false>(c, src, fc, f, i_begin, i_end, partials, req, finalized);
#endif
    }
    if constexpr (K == 3) {
        if (o.id == VS_OBJ_ISHIGAMI) {
            IshigamiReg<K> f{hp[0], hp[1]};
            if (second) return launch_fused_t<K, IshigamiReg<K>, true, false>(c, src, fc, f, i_begin, i_end, partials, req, finalized);
            return launch_fused_t<K, IshigamiReg<K>, false, false>(c, src, fc, f, i_begin, i_end, partials, req, finalized);
        }
    }
    set_error("objective %d has no fused kernel for k=%d", o.id, K);
    return VS_ERR_UNSUPPORTED;
}

// The one-launch step (estimators / peer exchange / chunk flags in the kernel's tail) exists for the warp-specialised variants.
template <int K>
static bool tail_supported_k(const vs_ctx *c, int flags) {
    const int v = fused_variant_for<K>(c, (flags & VS_FLAG_SECOND_ORDER) != 0, (flags & VS_FLAG_SEPARABLE) != 0, 0, false);
    return v == 5 || v == 6;     // (5 and 6 both have the tail: the choice between them does not matter here)
}

}  // namespace vs
