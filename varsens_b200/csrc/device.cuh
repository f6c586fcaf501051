// Device building blocks: Halton radical inverse, scaling, objective functors.
#pragma once

#include "vs_internal.cuh"

namespace vs {

// ---------------------------------------------------------------------------------------------
// Inline PTX shared by the kernels: shared-window addresses, mbarriers, the FP64 tensor MMA, the global timer.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// hint_ns: suspend-time hint of try_wait -- the warp sleeps in hardware instead of spinning
constexpr uint32_t MBAR_HINT_NS = 0x989680u;   // the fused and Gram kernels' hint (the export kernel passes a shorter one)
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity, uint32_t hint_ns) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity), "r"(hint_ns)
        : "memory");
}
// mma.sync m8n8k4 f64: {c0, c1} += a * b (one A and one B element per lane)
__device__ __forceinline__ void dmma_m8n8k4(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// ---------------------------------------------------------------------------------------------
// Halton: ghalton's in-order digit sum (call sites varsens/saltelli.py:82-84; SURVEY.md App. C).
//   x = 0; for j = 0.. (least-significant digit first): x += digit_j / b^(j+1)
// digit_j / b^(j+1) is read from the host-built table, so the device performs exactly the same
// sequence of IEEE additions as the CPU statement and no fp64 division.  __dadd_rn forbids any
// re-association / contraction.  Base 2 is exact in every partial sum, hence a bit reversal.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double radical_inverse(const double *__restrict__ T, uint32_t b, uint64_t magic, uint32_t m) {
    if (b == 2u) return (double)__brev(m) * 2.3283064365386962890625e-10;  // 2^-32, exact
    double x = 0.0;
    while (m != 0u) {
        uint32_t q = (uint32_t)__umul64hi((uint64_t)m, magic);
        uint32_t d = m - q * b;
        x = __dadd_rn(x, T[d]);
        T += b;
        m = q;
    }
    return x;
}

// VS_HALTON_HORNER: x = (x + digit_j) / b from the most significant digit down (one fp64 division per digit).
// Digits are kept in 32 bits: from dimension 54 on the bases exceed 255 (the 55th prime is 257).
__device__ __forceinline__ double radical_inverse_horner(uint32_t b, uint64_t magic, uint32_t m) {
    if (b == 2u) return (double)__brev(m) * 2.3283064365386962890625e-10;
    uint32_t dig[32];
    int nd = 0;
    while (m != 0u) {
        uint32_t q = (uint32_t)__umul64hi((uint64_t)m, magic);
        dig[nd++] = m - q * b;
        m = q;
    }
    double x = 0.0;
    const double bd = (double)b;
    for (int j = nd - 1; j >= 0; --j) x = __ddiv_rn(__dadd_rn(x, (double)dig[j]), bd);
    return x;
}

__device__ __forceinline__ double halton_coord(const HaltonDev &h, int d, uint32_t m) {
    if (h.mode == VS_HALTON_HORNER) return radical_inverse_horner(h.base[d], h.magic[d], m);
    return radical_inverse(h.terms + h.off[d], h.base[d], h.magic[d], m);
}

// ---------------------------------------------------------------------------------------------
// Multiply-only digit loop for kernels with RUN-TIME bases (export mode, product-form evaluation): lane = base row, the
// whole warp walks one dimension, the A chain and the B chain of a row advance together.  Per dimension (warp-uniform):
//   nd  digit positions of the launch's largest index (an exhausted index keeps adding the term of digit 0 = 0.0: exact),
//       so the loop has a fixed trip count -- no per-step "any lane left?" test, nothing for the compiler to predicate;
//   jg  leading positions that need the general division (64-bit magic mul-high), until m * 8b < 2^32 holds for every
//       index of the launch; from there on  w = m * ceil(2^32 / b):  quotient = hi(w),  8 * digit = umulhi(lo(w), 8b)
//       (two multiplies; proof and brute-force check: tools/check_fastdiv.py, the same step as fused_impl.cuh: digit_step).
// The term of a digit is read from the shared-memory table (TABLE: row address + 8 * digit is the byte address), or
// computed as fma(dd, rh, dd * rl), dd = 8 * digit -- the product with a double-double reciprocal, bit-equal to the table
// entry (host.cu: build_arith checks every digit of every position and clears arith_ok otherwise).
// ---------------------------------------------------------------------------------------------
struct DimLoop {
    uint32_t b8, c32;
    int nd, jg;
};

__device__ __forceinline__ DimLoop dim_loop(uint32_t b, uint64_t max_index) {
    DimLoop dl;
    dl.b8 = 8u * b;
    dl.c32 = (uint32_t)((0x100000000ull + b - 1) / b);
    dl.nd = 0;
    dl.jg = 0;
    for (uint64_t m = max_index; m > 0; m /= b) {
        if (m * 8ull * b >= 0x100000000ull) dl.jg = dl.nd + 1;
        ++dl.nd;
    }
    return dl;
}

// NR row groups per lane: the lane's rows r, r + 32, ... advance together (2 NR chains per dimension) with the SAME
// warp-uniform constants -- the per-dimension prologue is paid once for NR rows and the independent work per warp grows NR-fold.
template <bool TABLE, int NR>
__device__ __forceinline__ void halton_pair(const uint32_t (&ia)[NR], const uint32_t (&ib)[NR], uint32_t b, uint64_t magic,
                                            const DimLoop dl, uint32_t row, const double *__restrict__ rh,
                                            const double *__restrict__ rl, double (&pa)[NR], double (&pb)[NR]) {
    auto term = [&](uint32_t off8, int j) -> double {
        if constexpr (TABLE) {
            double t;
            asm("ld.shared.f64 %0, [%1];" : "=d"(t) : "r"(row + off8));
            return t;
        } else {
            const double dd = __dadd_rn(__hiloint2double(0x43300000, (int)off8), -4503599627370496.0);   // 2^52 + off8, exact
            return __fma_rn(dd, rh[j], __dmul_rn(dd, rl[j]));
        }
    };
    uint32_t ma[NR], mb[NR];
#pragma unroll
    for (int r = 0; r < NR; ++r) { ma[r] = ia[r]; mb[r] = ib[r]; pa[r] = 0.0; pb[r] = 0.0; }
    int j = 0;
#pragma unroll 1
    for (; j < dl.jg; ++j) {                                  // usually 0 or 1 trips
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const uint32_t qa = (uint32_t)__umul64hi((uint64_t)ma[r], magic), qb = (uint32_t)__umul64hi((uint64_t)mb[r], magic);
            pa[r] = __dadd_rn(pa[r], term(8u * (ma[r] - qa * b), j));
            pb[r] = __dadd_rn(pb[r], term(8u * (mb[r] - qb * b), j));
            ma[r] = qa;
            mb[r] = qb;
        }
        if constexpr (TABLE) row += dl.b8;
    }
#pragma unroll(NR == 1 ? 2 : 1)
    for (; j < dl.nd; ++j) {
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const uint64_t wa = (uint64_t)ma[r] * dl.c32, wb = (uint64_t)mb[r] * dl.c32;
            ma[r] = (uint32_t)(wa >> 32);
            mb[r] = (uint32_t)(wb >> 32);
            pa[r] = __dadd_rn(pa[r], term(__umulhi((uint32_t)wa, dl.b8), j));
            pb[r] = __dadd_rn(pb[r], term(__umulhi((uint32_t)wb, dl.b8), j));
        }
        if constexpr (TABLE) row += dl.b8;
    }
}

// Two dimensions with computed terms at once: 4 NR chains (A and B index of NR rows in dimensions d1 and d2) share one
// loop -- half the loop and branch overhead per dimension and twice the independent work per warp.  The trip counts are
// the larger ones of the two dimensions: a general division step is exact for any index, and a position beyond a
// dimension's last digit adds fma(0, rh, 0 * rl) = +0.0.
template <int NR>
__device__ __forceinline__ void halton_quad_arith(const uint32_t (&ia)[NR], const uint32_t (&ib)[NR], uint32_t b1, uint64_t magic1,
                                                  const DimLoop dl1, const double *__restrict__ rh1, const double *__restrict__ rl1,
                                                  uint32_t b2, uint64_t magic2, const DimLoop dl2, const double *__restrict__ rh2,
                                                  const double *__restrict__ rl2, double (&pa1)[NR], double (&pb1)[NR],
                                                  double (&pa2)[NR], double (&pb2)[NR]) {
    auto term = [](uint32_t off8, double rh, double rl) -> double {
        const double dd = __dadd_rn(__hiloint2double(0x43300000, (int)off8), -4503599627370496.0);       // 2^52 + off8, exact
        return __fma_rn(dd, rh, __dmul_rn(dd, rl));
    };
    uint32_t ma1[NR], mb1[NR], ma2[NR], mb2[NR];
#pragma unroll
    for (int r = 0; r < NR; ++r) {
        ma1[r] = ia[r]; mb1[r] = ib[r]; ma2[r] = ia[r]; mb2[r] = ib[r];
        pa1[r] = 0.0; pb1[r] = 0.0; pa2[r] = 0.0; pb2[r] = 0.0;
    }
    const int jg = max(dl1.jg, dl2.jg), nd = max(dl1.nd, dl2.nd);
    int j = 0;
#pragma unroll 1
    for (; j < jg; ++j) {                                     // usually 0 or 1 trips
        const double h1 = rh1[j], l1 = rl1[j], h2 = rh2[j], l2 = rl2[j];
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const uint32_t qa1 = (uint32_t)__umul64hi((uint64_t)ma1[r], magic1), qb1 = (uint32_t)__umul64hi((uint64_t)mb1[r], magic1);
            const uint32_t qa2 = (uint32_t)__umul64hi((uint64_t)ma2[r], magic2), qb2 = (uint32_t)__umul64hi((uint64_t)mb2[r], magic2);
            pa1[r] = __dadd_rn(pa1[r], term(8u * (ma1[r] - qa1 * b1), h1, l1));
            pb1[r] = __dadd_rn(pb1[r], term(8u * (mb1[r] - qb1 * b1), h1, l1));
            pa2[r] = __dadd_rn(pa2[r], term(8u * (ma2[r] - qa2 * b2), h2, l2));
            pb2[r] = __dadd_rn(pb2[r], term(8u * (mb2[r] - qb2 * b2), h2, l2));
            ma1[r] = qa1; mb1[r] = qb1; ma2[r] = qa2; mb2[r] = qb2;
        }
    }
#pragma unroll 1
    for (; j < nd; ++j) {
        const double h1 = rh1[j], l1 = rl1[j], h2 = rh2[j], l2 = rl2[j];
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const uint64_t wa1 = (uint64_t)ma1[r] * dl1.c32, wb1 = (uint64_t)mb1[r] * dl1.c32;
            const uint64_t wa2 = (uint64_t)ma2[r] * dl2.c32, wb2 = (uint64_t)mb2[r] * dl2.c32;
            ma1[r] = (uint32_t)(wa1 >> 32); mb1[r] = (uint32_t)(wb1 >> 32);
            ma2[r] = (uint32_t)(wa2 >> 32); mb2[r] = (uint32_t)(wb2 >> 32);
            pa1[r] = __dadd_rn(pa1[r], term(__umulhi((uint32_t)wa1, dl1.b8), h1, l1));
            pb1[r] = __dadd_rn(pb1[r], term(__umulhi((uint32_t)wb1, dl1.b8), h1, l1));
            pa2[r] = __dadd_rn(pa2[r], term(__umulhi((uint32_t)wa2, dl2.b8), h2, l2));
            pb2[r] = __dadd_rn(pb2[r], term(__umulhi((uint32_t)wb2, dl2.b8), h2, l2));
        }
    }
}

// Shared-memory constants of the run-time-base generators (export mode, product-form evaluation), filled once per CTA
// (halton_prefix).  HL_D0, HL_J: vs_internal.cuh.
struct HaltonShared {
    const uint32_t *base, *off;
    const uint64_t *magic;
    const DimLoop *dl;
    const double *arh, *arl;
    uint32_t table_saddr;      // shared-window byte address of the table prefix (dimensions < HL_D0)
};

// The unscaled coordinates of one row pair (A index ia, B index ib), lane = row, distributed over the warps of a team by
// UNITS: unit u < min(k, HL_D0) is the single dimension u (base 2: a bit reversal; bases 3..31: table terms), the units after
// those are PAIRS of computed-term dimensions (HL_D0 + 2p, HL_D0 + 2p + 1).  ulist[w * HL_MAXQ + q] is the q-th unit of warp w,
// 255 ends the list (halton_schedule); emit receives every coordinate once.  All branches are warp-uniform.
constexpr int HL_MAXQ = 32;            // units per warp at most
constexpr int HL_MAX_UNITS = 160;      // k <= 309: at most 20 units per warp on average with 8 warps
constexpr int HL_LIST_BYTES = 16 * HL_MAXQ;   // up to 16 warps
__host__ __device__ inline int halton_unit_count(int k) {
    const int nsmall = k < HL_D0 ? k : HL_D0;
    return nsmall + (k - nsmall + 1) / 2;
}

// Longest-processing-time assignment of the units to `nw` warps (one thread, once per CTA).  A unit's cost is its digit
// count plus a fixed part (measured with per-dimension clock stamps in the export kernel: ~0.4 k cycles fixed, ~0.11 k per
// digit step of a two-chain loop, a four-chain pair step ~2.2x that).  Both unit lists are already in descending cost order
// (digit counts fall with the base), so a merge replaces the sort.  Round-robin assignment left the warps that own the base-3
// and base-5 dimensions with 5.0 k cycles per tile against an average of 2.9 k.
__device__ inline void halton_schedule(int k, int nw, const DimLoop *dl, unsigned char *ulist) {
    const int nsmall = k < HL_D0 ? k : HL_D0, nunits = halton_unit_count(k);
    float load[16];
    int cnt[16];
    for (int w = 0; w < nw; ++w) { load[w] = 0.0f; cnt[w] = 0; }
    for (int e = 0; e < nw * HL_MAXQ; ++e) ulist[e] = 255;
    auto cost_pair = [&](int u) {
        const int d1 = HL_D0 + 2 * (u - nsmall), d2 = d1 + 1;
        return d2 < k ? 4.0f + 2.2f * (float)max(dl[d1].nd, dl[d2].nd) : 4.0f + 1.2f * (float)dl[d1].nd;
    };
    auto place = [&](int u, float c) {
        int best = -1;
        for (int w = 0; w < nw; ++w)
            if (cnt[w] < HL_MAXQ - 1 && (best < 0 || load[w] < load[best])) best = w;
        load[best] += c;
        ulist[best * HL_MAXQ + cnt[best]++] = (unsigned char)u;
    };
    int is = 1, ip = nsmall;
    while (is < nsmall || ip < nunits) {
        const float cs = is < nsmall ? 4.0f + (float)dl[is].nd : -1.0f;
        const float cp = ip < nunits ? cost_pair(ip) : -1.0f;
        if (cs >= cp) place(is++, cs);
        else place(ip++, cp);
    }
    if (nunits > 0) place(0, 1.0f);                          // dimension 0: base 2, a bit reversal
}

// emit(d, r, pa, pb): coordinate d of the lane's r-th row (A point, B point).
template <int NR, class Emit>
__device__ __forceinline__ void halton_units(int w, const unsigned char *__restrict__ ulist, int k, const uint32_t (&ia)[NR],
                                             const uint32_t (&ib)[NR], const HaltonShared &hs, Emit &&emit) {
    const int nsmall = k < HL_D0 ? k : HL_D0;
    const uint32_t *wl = reinterpret_cast<const uint32_t *>(ulist + w * HL_MAXQ);      // four units per load
    uint32_t pack = wl[0];
    for (int q = 0;; ++q) {
        if (q && (q & 3) == 0) pack = wl[q >> 2];
        const int u = (int)(pack & 255u);
        pack >>= 8;
        if (u == 255) break;
        if (u < nsmall) {
            const uint32_t b = hs.base[u];
            double pa[NR], pb[NR];
            if (b == 2u) {
#pragma unroll
                for (int r = 0; r < NR; ++r) {
                    pa[r] = (double)__brev(ia[r]) * 2.3283064365386962890625e-10;
                    pb[r] = (double)__brev(ib[r]) * 2.3283064365386962890625e-10;
                }
            } else {
                halton_pair<true, NR>(ia, ib, b, hs.magic[u], hs.dl[u], hs.table_saddr + 8u * hs.off[u], nullptr, nullptr, pa, pb);
            }
#pragma unroll
            for (int r = 0; r < NR; ++r) emit(u, r, pa[r], pb[r]);
        } else {
            const int d1 = HL_D0 + 2 * (u - nsmall), d2 = d1 + 1;
            if (d2 < k) {
                double pa1[NR], pb1[NR], pa2[NR], pb2[NR];
                halton_quad_arith<NR>(ia, ib, hs.base[d1], hs.magic[d1], hs.dl[d1], hs.arh + (size_t)d1 * HL_J, hs.arl + (size_t)d1 * HL_J,
                                      hs.base[d2], hs.magic[d2], hs.dl[d2], hs.arh + (size_t)d2 * HL_J, hs.arl + (size_t)d2 * HL_J, pa1,
                                      pb1, pa2, pb2);
#pragma unroll
                for (int r = 0; r < NR; ++r) { emit(d1, r, pa1[r], pb1[r]); emit(d2, r, pa2[r], pb2[r]); }
            } else {
                double pa[NR], pb[NR];
                halton_pair<false, NR>(ia, ib, hs.base[d1], hs.magic[d1], hs.dl[d1], 0u, hs.arh + (size_t)d1 * HL_J, hs.arl + (size_t)d1 * HL_J,
                                       pa, pb);
#pragma unroll
                for (int r = 0; r < NR; ++r) emit(d1, r, pa[r], pb[r]);
            }
        }
    }
}

// The generator prefix of a run-time-base kernel's shared memory:
//   base[k] off[k] (u32) | magic[k] (u64) | lb[k] wr[k] | dl[k] | arh arl [k][HL_J] | ulist[16][HL_MAXQ] (u8) | table[table_len]
// halton_prefix_doubles: the doubles before the table (20 k + 64, even: a 16-byte aligned prefix with an even table_len ends
// 16-byte aligned).
__host__ __device__ constexpr size_t halton_prefix_doubles(int k) {
    return (2 * (size_t)k + 1) / 2 + (size_t)k + 2 * (size_t)k + 2 * (size_t)k + 2 * (size_t)k * HL_J + HL_LIST_BYTES / 8;
}
struct HaltonPrefix {
    HaltonShared hs;
    const unsigned char *ulist;
    const double *lb, *wr;     // scaling constants (0.0 / 1.0 under identity scaling)
    double *table;             // the table prefix
};
// Carves the prefix out of p and fills it; every thread of the CTA calls it, it ends with __syncthreads.  Unless the points are
// given (src.raw): base, off, magic and the first table_len doubles of the term table; `computed`: also dl, arh and arl (the
// multiply-only digit loop and the computed terms); sched_warps > 0: the units of that many warps (halton_schedule).
__device__ __forceinline__ HaltonPrefix halton_prefix(double *p, int k, const SourceDev &src, const ScaleDev &s, uint32_t table_len,
                                                      bool computed, int sched_warps) {
    uint32_t *base = reinterpret_cast<uint32_t *>(p), *off = base + k;
    uint64_t *magic = reinterpret_cast<uint64_t *>(p + (2 * k + 1) / 2);
    double *lb = reinterpret_cast<double *>(magic + k), *wr = lb + k;
    DimLoop *dl = reinterpret_cast<DimLoop *>(wr + k);                 // 16 bytes per dimension
    double *arh = reinterpret_cast<double *>(dl + k), *arl = arh + (size_t)k * HL_J;
    unsigned char *ulist = reinterpret_cast<unsigned char *>(arl + (size_t)k * HL_J);
    double *table = arl + (size_t)k * HL_J + HL_LIST_BYTES / 8;
    const int tid = threadIdx.x, nthr = blockDim.x;
    if (!src.raw) {
        for (int d = tid; d < k; d += nthr) {
            base[d] = src.h.base[d];
            off[d] = src.h.off[d];
            magic[d] = src.h.magic[d];
            if (computed) dl[d] = dim_loop(src.h.base[d], src.start + 2 * src.n - 1);      // the largest index of the design
        }
        if (computed)
            for (int e = tid; e < k * HL_J; e += nthr) { arh[e] = src.h.arh[e]; arl[e] = src.h.arl[e]; }
        for (uint32_t e = tid; e < table_len; e += nthr) table[e] = src.h.terms[e];
    }
    for (int d = tid; d < k; d += nthr) {
        lb[d] = s.kind != VS_SCALE_IDENTITY ? s.lb[d] : 0.0;
        wr[d] = s.kind != VS_SCALE_IDENTITY ? s.wr[d] : 1.0;
    }
    __syncthreads();
    if (sched_warps > 0 && tid == 0) halton_schedule(k, sched_warps, dl, ulist);
    __syncthreads();
    return {{base, off, magic, dl, arh, arl, smem_u32(table)}, ulist, lb, wr, table};
}

// ---------------------------------------------------------------------------------------------
// scale.py:33 (two roundings: multiply, then add -- never an FMA) and :62.  The one device statement of both.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double scale_value(int kind, double lb, double wr, double p) {
    if (kind == VS_SCALE_LINEAR) return __dadd_rn(__dmul_rn(p, wr), lb);
    if (kind == VS_SCALE_POWER) return __dmul_rn(lb, pow(wr, p));
    return p;
}
// s.lb and s.wr are null under identity scaling: read in the branch of their kind only
__device__ __forceinline__ double apply_scale(const ScaleDev &s, int d, double p) {
    if (s.kind == VS_SCALE_LINEAR) return scale_value(VS_SCALE_LINEAR, s.lb[d], s.wr[d], p);
    if (s.kind == VS_SCALE_POWER) return scale_value(VS_SCALE_POWER, s.lb[d], s.wr[d], p);
    return p;
}

// Unscaled coordinate d of A_i / B_i (SURVEY.md App. A):
//   A_i = h(start + i),  B_i = h(start + n + perm[i])      (or the rows of `raw`)
__device__ __forceinline__ double source_a(const SourceDev &src, int k, uint64_t i, int d) {
    if (src.raw) return src.raw[i * (uint64_t)k + d];
    return halton_coord(src.h, d, (uint32_t)(src.start + i));
}
__device__ __forceinline__ double source_b(const SourceDev &src, int k, uint64_t pi, int d) {
    if (src.raw) return src.raw[(src.n + pi) * (uint64_t)k + d];
    return halton_coord(src.h, d, (uint32_t)(src.start + src.n + pi));
}

// ---------------------------------------------------------------------------------------------
// Objective functors.  X is any type with `double operator[](int) const` (registers, shared
// memory view, ...).  params layout on the device (built by get_objective):
//   GFUNCTION : [0,k) a_c        [k,2k) 1/(1+a_c)      [2k,3k) a_c/(1+a_c)
//   ISHIGAMI  : A, B
//   RK4_CHAIN : dt, nsteps
// ---------------------------------------------------------------------------------------------
struct GFunction {
    const double *inv;   // 1/(1+a_c)
    const double *off;   // a_c/(1+a_c)
    static constexpr bool product_form = true;           // f(x) = prod_c term(c, x_c), evaluated in ascending c from 1.0
    __device__ __forceinline__ double term(int c, double x) const {
        double t = fma(4.0, x, -2.0);                     // 4x - 2         (2 flops)
        return fma(fabs(t), inv[c], off[c]);              // (|t| + a)/(1+a) (2)
    }
    template <class X>
    __device__ __forceinline__ double operator()(const X &x, int k) const {
        double p = 1.0;
        for (int c = 0; c < k; ++c) p *= term(c, x[c]);   // running product (1)
        return p;
    }
};

struct Ishigami {
    double A, B;
    template <class X>
    __device__ __forceinline__ double operator()(const X &x, int) const {
        double s0 = sin(x[0]), s1 = sin(x[1]), x2 = x[2];
        double x22 = x2 * x2;
        return s0 + A * s1 * s1 + B * (x22 * x22) * s0;
    }
};

// Reversible chain, S links, S+1 species.  Register-resident for compile-time S.
// FROZEN ARITHMETIC (the oracle, oracle/oracle.c: f_rk4_chain, performs exactly these roundings, so trajectories are
// bit-identical given bit-identical rate constants): every product-sum below is ONE fused multiply-add where written as
// fma(), one rounded multiply / add / subtract where written as __dmul_rn / __dadd_rn / __dsub_rn; nothing is left to the
// compiler's contraction choices.
//   flux_s = fma(kf_s, X_s, -(kr_s * X_{s+1}))     d_s = flux_{s-1} - flux_s
//   stage  : T = fma(h, d, X)                       sum: a = k1, a = fma(2, k2, a), a = fma(2, k3, a), a = a + k4
//   update : X = fma(dt/6, a, X)
// (This is what nvcc's default contraction produced before it was pinned: the change cost nothing -- C5 runs at the same
// 71 % of the FP64 peak.)
template <int S>
struct RK4Chain {
    double dt;
    int nsteps;
    __device__ __forceinline__ static void rhs(const double (&X)[S + 1], const double (&kf)[S], const double (&kr)[S],
                                               double (&d)[S + 1]) {
        double prev = 0.0;
#pragma unroll
        for (int s = 0; s < S; ++s) {
            double flux = fma(kf[s], X[s], -__dmul_rn(kr[s], X[s + 1]));
            d[s] = __dsub_rn(prev, flux);
            prev = flux;
        }
        d[S] = prev;
    }
    template <class XV>
    __device__ __forceinline__ double operator()(const XV &x, int) const {
        double kf[S], kr[S], X[S + 1], T[S + 1], a[S + 1], d[S + 1];
#pragma unroll
        for (int s = 0; s < S; ++s) { kf[s] = x[s]; kr[s] = x[S + s]; }
#pragma unroll
        for (int s = 0; s <= S; ++s) X[s] = 0.0;
        X[0] = 1.0;
        const double h2 = __dmul_rn(0.5, dt), h6 = __ddiv_rn(dt, 6.0);
        for (int it = 0; it < nsteps; ++it) {
            rhs(X, kf, kr, d);                                   // k1
#pragma unroll
            for (int s = 0; s <= S; ++s) { a[s] = d[s]; T[s] = fma(h2, d[s], X[s]); }
            rhs(T, kf, kr, d);                                   // k2
#pragma unroll
            for (int s = 0; s <= S; ++s) { a[s] = fma(2.0, d[s], a[s]); T[s] = fma(h2, d[s], X[s]); }
            rhs(T, kf, kr, d);                                   // k3
#pragma unroll
            for (int s = 0; s <= S; ++s) { a[s] = fma(2.0, d[s], a[s]); T[s] = fma(dt, d[s], X[s]); }
            rhs(T, kf, kr, d);                                   // k4
#pragma unroll
            for (int s = 0; s <= S; ++s) X[s] = fma(h6, __dadd_rn(a[s], d[s]), X[s]);
        }
        return X[S];
    }
};

// Run-time S (any k): state in local memory.  Same frozen arithmetic as RK4Chain<S>.
struct RK4ChainDyn {
    double dt;
    int nsteps;
    static constexpr int MAXS = 64;
    template <class XV>
    __device__ double operator()(const XV &x, int k) const {
        const int S = k / 2;
        double X[MAXS + 1], T[MAXS + 1], a[MAXS + 1], d[MAXS + 1];
        for (int s = 0; s <= S; ++s) X[s] = 0.0;
        X[0] = 1.0;
        const double h2 = __dmul_rn(0.5, dt), h6 = __ddiv_rn(dt, 6.0);
        auto rhs = [&](const double *Y) {
            double prev = 0.0;
            for (int s = 0; s < S; ++s) {
                double flux = fma(x[s], Y[s], -__dmul_rn(x[S + s], Y[s + 1]));
                d[s] = __dsub_rn(prev, flux);
                prev = flux;
            }
            d[S] = prev;
        };
        for (int it = 0; it < nsteps; ++it) {
            rhs(X);
            for (int s = 0; s <= S; ++s) { a[s] = d[s]; T[s] = fma(h2, d[s], X[s]); }
            rhs(T);
            for (int s = 0; s <= S; ++s) { a[s] = fma(2.0, d[s], a[s]); T[s] = fma(h2, d[s], X[s]); }
            rhs(T);
            for (int s = 0; s <= S; ++s) { a[s] = fma(2.0, d[s], a[s]); T[s] = fma(dt, d[s], X[s]); }
            rhs(T);
            for (int s = 0; s <= S; ++s) X[s] = fma(h6, __dadd_rn(a[s], d[s]), X[s]);
        }
        return X[S];
    }
};

// MassAction (VS_OBJ_MASS_ACTION, a run-time network; kernel in kernels_network.cu).  FROZEN ARITHMETIC, restated by the
// oracle (oracle/mass_action.c: ma_rhs, f_mass_action) so trajectories are bit-identical given bit-identical rates and initial amounts:
//   P      = 1.0 (no species on the side), X[s0] (one), __dmul_rn(X[s0], X[s1]) (two)      Pf over reactants, Pr over products
//   flux_r = fma(kf, Pf, -__dmul_rn(kr, Pr))   reversible;   __dmul_rn(kf, Pf)   irreversible (reverse term not evaluated)
//   d_s    = 0.0, then over the reactions with net coefficient c != 0 for s (products - reactants; a catalyst nets to 0),
//            ascending:  c = +1: __dadd_rn(d, flux)   c = -1: __dsub_rn(d, flux)   |c| = 2: fma(c, flux, d)
//   stages and update exactly RK4Chain's (h2 = 0.5*dt, h6 = dt/6, T = fma(h, d, X), a = k1, a = fma(2, k2, a),
//            a = fma(2, k3, a), X = fma(h6, __dadd_rn(a, k4), X))
//   observable o: acc = 0.0, acc = fma(w[o][s], X_s, acc) over the nonzero weights, ascending s.
// The chain written as a network (X_s <-> X_{s+1}, kf = x[s], kr = x[S+s], X(0) = e_0, observable X_S) therefore yields the
// same bits as RK4Chain<S> and RK4ChainDyn.

// MassActionAdaptive (VS_OBJ_MASS_ACTION_ADAPTIVE; kernel network_adaptive_kernel in kernels_network.cu).  FROZEN ARITHMETIC,
// restated bit for bit by the oracle (oracle/mass_action.c: f_mass_action_adaptive).  Only correctly rounded operations
// (+ - * /, fma, sqrt, fabs, fmax, fmin): CUDA and glibc round pow, exp and log differently, so the step-size controller uses
// none of them.
//   right-hand side   MassAction's P, flux_r and d_s above.
//   tableau           Dormand-Prince 5(4), Hairer-Norsett-Wanner I, Table 5.2: a_ij, and e_j = b_j - bhat_j, each the
//                     correctly rounded double of its rational (dp5:: in kernels_network.cu).
//   start             t = 0.0, h = h0, K1 = f(X).  attempts = 0.
//   attempt           to = the next output time; hs = h, or hs = to - t (clipped) if t + h >= to.  If attempts == max_steps,
//                     or t + hs == t: the trajectory has failed, outputs of this and every later time are NaN, stop.
//                     Else attempts += 1 and, for stage i = 2..7: acc = 0.0, acc = fma(a_ij, K_j[s], acc) over the j with
//                     a_ij != 0, ascending; Y[s] = fma(hs, acc, X[s]); K_i = f(Y).  Y after stage 7 is the 5th-order
//                     solution, K7 = f(Y) (stored in K2's slot).
//   error             E_s = hs * (fma chain of e_j K_j[s] from 0.0, j = 1, 3, 4, 5, 6, 7);  sc_s = fma(rtol, fmax(|X_s|, |Y_s|),
//                     atol);  r = E_s / sc_s;  q = fma(r, r, q) from 0.0 over ascending s;  err = sqrt(q / S).
//   controller        fac_max = 1.0 on the attempt after a rejection, else 5.0.  fac = fac_max if err == 0; 0.2 if err is
//                     not finite; else fmin(fac_max, fmax(0.2, 0.9 / sqrt(sqrt(err)))).  (Exponent 1/4 rather than the
//                     textbook 1/5: two square roots.)
//   accept iff err <= 1.0:  t = to if clipped, else t + hs;  X = Y;  K1 = K7 (FSAL: each attempt costs 6 right-hand sides,
//                     the first step 7; a rejected attempt keeps K1).  At a clipped step the L observables at `to` are
//                     MassAction's: acc = fma(w[o][s], X_s, acc) from 0.0 over the nonzero weights, ascending s.
//   next step         h = hs * fac (accepted or not).

// MassActionStiff (VS_OBJ_MASS_ACTION_STIFF; kernel network_rosenbrock_kernel in kernels_network.cu).  FROZEN ARITHMETIC,
// restated bit for bit by the oracle (oracle/mass_action_stiff.c: f_mass_action_stiff), same operation rules as MassActionAdaptive.
// Rodas3 (Sandu et al. 1997, as tabulated in KPP's Rosenbrock.f90), autonomous form, gamma = 1/2, G = I/(hs gamma) - J(X):
//   right-hand side   MassAction's.  f(X) is kept across rejected attempts and formed again after each accepted step.
//   start, attempt    MassActionAdaptive's: t, h = h0, output-time clipping, max_steps, t + hs == t (NaN from there on).
//   Jacobian, factor  the slots of the factor's pattern (kernels_network.cu: stiff_program) are set to 0.0; then, over the
//                     reactions ascending, for each of its columns c (reactants, and products if reversible; catalysts
//                     included): dP = d(side product)/dX_c (0, 1, X_other, or 2 * X_c for a homodimer), d = fma(kf, dPf,
//                     -(kr * dPr)) if reversible else kf * dPf, and for each species s with net coefficient nu != 0:
//                     G[s][c] = fma(-nu, d, G[s][c]).  Then G[s][s] += 1 / (0.5 * hs).  Then right-looking LU without
//                     pivoting in elimination order p = 0 .. S-1: a pivot that is 0 or not finite rejects the attempt with
//                     h = hs * 0.2 (the trajectory goes on, the next attempt is "after a rejection"); else for each L entry
//                     (i, p): l = G[i][p] / pivot, G[i][p] = l, and for each U entry (p, j): G[i][j] = fma(-l, G[p][j], G[i][j]).
//   solve             b = G^{-1} b in place: forward, p ascending, b[i] = fma(-L[i][p], b[p], b[i]) over L entries (i, p);
//                     back, p descending, acc = b[p], acc = fma(-U[p][j], b[j], acc) over U entries (p, j), j ascending in
//                     elimination position, b[p] = acc / U[p][p].
//   stages            c_ij = C_ij / hs (C21 = 4, C31 = 1, C32 = -1, C41 = 1, C42 = -1, C43 = -8/3 correctly rounded).
//                     K1 = solve(f(X));  K2 = solve(fma(c21, K1, f(X)));  Y = fma(2, K1, X);
//                     K3 = solve(fma(c32, K2, fma(c31, K1, f(Y))));  Y = Y + K3;
//                     K4 = solve(fma(c43, K3, fma(c42, K2, fma(c41, K1, f(Y)))));  X_new = Y + K4 (stiffly accurate).
//   error             sc_s = fma(rtol, fmax(|X_s|, |X_new,s|), atol);  r = K4_s / sc_s;  q = fma(r, r, q) from 0.0 over
//                     ascending s;  err = sqrt(q / S).
//   controller        fac_max = 1.0 on the attempt after a rejection, else 6.0.  fac = 0.2 if err is not finite; else
//                     fmin(fac_max, fmax(0.2, 0.9 / cbrt(fmin(fmax(err, 1e-3), 1e3)))) (the clamp changes no factor: outside
//                     it the bounds apply), where cbrt(a) = four Newton steps y = fma(2, y, a / (y * y)) / 3 from the bits
//                     (bits(a) / 3 + 0x2A9F7893782DA1CE) as an unsigned 64-bit integer division.
//   accept iff err <= 1.0:  t = to if clipped, else t + hs;  X = X_new; observables at a clipped step as MassActionAdaptive.
//   next step         h = hs * fac (accepted or not).

__host__ __device__ __forceinline__ void tile_coords(int id, int nt, int &tr, int &tc) {
    tr = 0;
    int rowlen = nt;
    while (id >= rowlen) { id -= rowlen; --rowlen; ++tr; }
    tc = tr + id;
}

// ---------------------------------------------------------------------------------------------
// Finalisation: the estimators of varsens/saltelli.py:577-622 on the sufficient statistics, same
// operation order (E_2 over n; U and Grams over n-1; mixed normalisation is the reference's).
// Called by every thread of ONE CTA (finalize_kernel, the peer-memory exchange kernel, the tail of the
// fused kernel).  P = packed partial sums (vs_partials_len), res = result vector:
// E_2[l] var_y[l] U_j[kl] U_nj[kl] sens[kl] sens_t[kl] sens_2[(kl)^2] sens_2n[(kl)^2]
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double gram_at(const double *G, int m, int p, int q) {
    if (p > q) { int t = p; p = q; q = t; }
    return G[(size_t)p * m - (size_t)p * (p - 1) / 2 + (size_t)(q - p)];
}

__device__ __forceinline__ void finalize_body(int k, int l, double n, double rows, const double *__restrict__ P, int second_order,
                              double *__restrict__ res) {
    const int m = (2 + 2 * k) * l;
    const double *G = P + 4 * l;
    const int kl = k * l;
    double *E2 = res, *var = res + l, *Uj = res + 2 * l, *Unj = Uj + kl, *sens = Unj + kl, *senst = sens + kl;
    double *s2 = senst + kl, *s2n = s2 + (size_t)kl * kl;
    __shared__ double sE2[64], sVar[64];
    for (int o = threadIdx.x; o < l; o += blockDim.x) {
        double e2 = gram_at(G, m, 0 * l + o, 1 * l + o) / n;                                  // :577
        double tot = P[o] + P[l + o];
        double v = (P[2 * l + o] + P[3 * l + o] - tot * tot / (2.0 * rows)) / (2.0 * rows - 1.0);   // :583 (ddof=1 over 2*rows values)
        E2[o] = e2;
        var[o] = v;
        if (o < 64) { sE2[o] = e2; sVar[o] = v; }
    }
    __syncthreads();
    auto e2_of = [&](int o) { return o < 64 ? sE2[o] : E2[o]; };
    auto var_of = [&](int o) { return o < 64 ? sVar[o] : var[o]; };
    for (int e = threadIdx.x; e < kl; e += blockDim.x) {
        int j = e / l, o = e - j * l;
        int iA = o, iB = l + o, iJ = (2 + j) * l + o, iN = (2 + k + j) * l + o;
        double uj = gram_at(G, m, iA, iJ) / (n - 1.0);                                        // :591-593
        uj += gram_at(G, m, iB, iN) / (n - 1.0);
        uj /= 2.0;
        double unj = gram_at(G, m, iA, iN) / (n - 1.0);                                       // :594-596
        unj += gram_at(G, m, iB, iJ) / (n - 1.0);
        unj /= 2.0;
        Uj[e] = uj;
        Unj[e] = unj;
        sens[e] = (uj - e2_of(o)) / var_of(o);                                                // :608
        senst[e] = 1.0 - ((unj - e2_of(o)) / var_of(o));                                      // :609
    }
    if (!second_order) return;
    for (size_t e = threadIdx.x; e < (size_t)kl * kl; e += blockDim.x) {
        int ia = (int)(e / kl), jb = (int)(e % kl);
        int i = ia / l, a = ia - i * l, j = jb / l, b = jb - j * l;
        int Ji = (2 + i) * l + a, Ni = (2 + k + i) * l + a, Jj = (2 + j) * l + b, Nj = (2 + k + j) * l + b;
        double v2 = gram_at(G, m, Ni, Jj) + gram_at(G, m, Ji, Nj);                            // :612-613
        v2 /= 2.0 * (n - 1.0);
        v2 -= e2_of(b);
        v2 /= var_of(b);
        double v2n = gram_at(G, m, Ni, Nj) + gram_at(G, m, Ji, Jj);                           // :618-619
        v2n /= 2.0 * (n - 1.0);
        v2n -= e2_of(b);
        v2n /= var_of(b);
        s2[e] = v2;
        s2n[e] = v2n;
    }
}

// ---------------------------------------------------------------------------------------------
// All-reduce of the partial-sum vector over NVLink peer memory, low-latency protocol: no fence, no separate flag.
// Every double travels as ONE 16-byte store {lo, epoch, hi, epoch}: each 8-byte half carries its own tag and is written
// atomically, so a reader that sees both tags equal to the current epoch has the value (what NCCL's LL protocol relies on).
// Rank r's vector goes to slot r of every rank's buffer (set = epoch parity: a rank that is one step ahead cannot overwrite
// slots somebody is still reading); every rank sums the world slots in rank order -> identical bits everywhere.
// Exchange buffer of a rank: 2 sets x world slots x plen elements x 16 bytes, zero-initialised; epoch starts at 1.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void ll_store(void *dst, double v, unsigned epoch) {
    const unsigned lo = (unsigned)__double2loint(v), hi = (unsigned)__double2hiint(v);
    asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "r"(lo), "r"(epoch), "r"(hi), "r"(epoch) : "memory");
}
// one warp per peer: src[0..plen) -> slot `rank` of every peer's set
__device__ __forceinline__ void ll_push(const uint64_t *__restrict__ bufs, int world, int rank, unsigned epoch, int plen,
                                        const double *__restrict__ src) {
    const int set = (int)(epoch & 1u);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
    for (int r = warp; r < world; r += nwarp) {
        char *dst = reinterpret_cast<char *>(bufs[r]) + (((size_t)set * world + rank) * plen) * 16;
        for (int e = lane; e < plen; e += 32) ll_store(dst + (size_t)e * 16, src[e], epoch);
    }
}
// dst[e] = sum over ranks (rank order) of slot r element e of MY buffer; waits (bounded) for each element's tags.
// Returns false if some element did not arrive within timeout_ns (dst is then incomplete).
__device__ __forceinline__ bool ll_reduce(const uint64_t *__restrict__ bufs, int world, int rank, unsigned epoch, int plen,
                                          double *__restrict__ dst, unsigned long long timeout_ns) {
    const int set = (int)(epoch & 1u);
    const char *mine = reinterpret_cast<const char *>(bufs[rank]) + ((size_t)set * world * plen) * 16;
    const unsigned long long t0 = globaltimer_ns();
    bool ok = true;
    for (int e = threadIdx.x; e < plen; e += blockDim.x) {
        double s = 0.0;
        for (int r = 0; r < world; ++r) {
            const char *p = mine + ((size_t)r * plen + e) * 16;
            unsigned lo, f0, hi, f1;
            for (;;) {
                asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(lo), "=r"(f0), "=r"(hi), "=r"(f1) : "l"(p) : "memory");
                if (f0 == epoch && f1 == epoch) break;
                if (globaltimer_ns() - t0 > timeout_ns) { ok = false; break; }
            }
            if (!ok) break;
            s += __hiloint2double((int)hi, (int)lo);
        }
        dst[e] = s;
        if (!ok) break;
    }
    return ok;
}

// ---------------------------------------------------------------------------------------------
// reductions
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace vs
