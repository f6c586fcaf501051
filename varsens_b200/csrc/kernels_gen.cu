// Generators and export-mode sample assembly.
#include "device.cuh"
#include <vector>
#include <cstdio>

namespace vs {

// ---------------------------------------------------------------------------------------------
// K1: Halton points, row-major (count, k).  One element per thread; consecutive threads write
// consecutive doubles.  Replaces varsens/saltelli.py:82-84 (+ :92/:95 scaling).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) halton_kernel(int k, uint64_t first, uint64_t total, HaltonDev h, ScaleDev s,
                                                     double *__restrict__ out) {
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
        uint64_t row = e / (uint32_t)k;
        int d = (int)(e - row * (uint32_t)k);
        double p = halton_coord(h, d, (uint32_t)(first + row));
        out[e] = apply_scale(s, d, p);
    }
}

int launch_halton(vs_ctx *c, int k, uint64_t first, uint64_t count, const HaltonDev &h, const ScaleDev &s, double *out) {
    uint64_t total = count * (uint64_t)k;
    if (total == 0) return VS_OK;
    uint64_t want = (total + 255) / 256;
    int grid = (int)(want < (uint64_t)c->sm_count * 32 ? want : (uint64_t)c->sm_count * 32);
    halton_kernel<<<grid, 256, 0, c->stream>>>(k, first, total, h, s, out);
    c->launches++;
    VS_CUDA(cudaGetLastError());
    return VS_OK;
}

// ---------------------------------------------------------------------------------------------
// K2: Gray-code Sobol by direct indexing (skip-ahead): point m = XOR of V[d][b] over the set bits
// b of m ^ (m >> 1); value = x * 2^-32.  Replaces quantlib/sobolGen.cpp:47-63.
// quantize6: the reference pipes the points through `cout << double` (6 significant digits) and
// numpy.loadtxt; that round trip is reproduced exactly in integer arithmetic:
//   x = X / 2^32 -> decimal D * 10^-p with D = round_half_even(X * 10^p / 2^32) in [10^5, 10^6]
//   -> strtod = correctly rounded D / 10^p (one IEEE division, both operands exact).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double quantize_6sig(uint32_t X) {
    if (X == 0u) return 0.0;
    // p = number of decimals so that X*10^p/2^32 has 6 integer digits: x in [10^-e, 10^-(e-1)) -> p = 5 + e
    // 10^p * X < 10^(p) * 2^32; p <= 15 keeps the product below 2^96 -> use 128-bit via two 64-bit halves.
    const double x = (double)X * 2.3283064365386962890625e-10;
    int e = 1;                       // x in [0.1, 1) -> e = 1
    double lim = 0.1;
    while (x < lim && e < 11) { lim *= 0.1; ++e; }   // coarse; corrected below with exact integers
    unsigned __int128 num, den = ((unsigned __int128)1) << 32;
    uint64_t D;
    int p = 5 + e;
    for (;;) {
        unsigned __int128 pw = 1;
        for (int i = 0; i < p; ++i) pw *= 10;
        num = (unsigned __int128)X * pw;
        unsigned __int128 q = num / den, r = num - q * den;
        D = (uint64_t)q;
        unsigned __int128 half = den >> 1;
        if (r > half || (r == half && (D & 1ull))) ++D;
        if (D < 100000ull) { ++p; continue; }        // estimate of e was one too small
        if (D > 1000000ull) { --p; continue; }
        break;                                       // D == 10^6 is fine: prints as 1 followed by zeros
    }
    double pw10 = 1.0;
    for (int i = 0; i < p; ++i) pw10 *= 10.0;        // exact for p <= 22
    return __ddiv_rn((double)D, pw10);
}

__global__ void __launch_bounds__(256) sobol_kernel(int k, uint64_t first, uint64_t total, const uint32_t *__restrict__ V,
                                                    int quantize6, ScaleDev s, double *__restrict__ out) {
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
        uint64_t row = e / (uint32_t)k;
        int d = (int)(e - row * (uint32_t)k);
        uint32_t m = (uint32_t)(first + row);
        uint32_t g = m ^ (m >> 1), x = 0u;
        const uint32_t *v = V + (size_t)d * 32;
        while (g) {
            int b = __ffs(g) - 1;
            x ^= v[b];
            g &= g - 1;
        }
        double p = quantize6 ? quantize_6sig(x) : (double)x * 2.3283064365386962890625e-10;
        out[e] = apply_scale(s, d, p);
    }
}

int launch_sobol(vs_ctx *c, int k, uint64_t first, uint64_t count, const uint32_t *dir_dev, int quantize6, const ScaleDev &s,
                 double *out) {
    uint64_t total = count * (uint64_t)k;
    if (total == 0) return VS_OK;
    uint64_t want = (total + 255) / 256;
    int grid = (int)(want < (uint64_t)c->sm_count * 32 ? want : (uint64_t)c->sm_count * 32);
    sobol_kernel<<<grid, 256, 0, c->stream>>>(k, first, total, dir_dev, quantize6, s, out);
    c->launches++;
    VS_CUDA(cudaGetLastError());
    return VS_OK;
}

// ---------------------------------------------------------------------------------------------
// K3: export mode.  A CTA owns TI consecutive base rows: it generates A (M_1 rows) and B (shuffled
// M_2 rows) ONCE into shared memory (2 * TI * k radical inverses) and then streams the 2+2k flat
// blocks that contain those rows -- each a contiguous TI*k-double run in HBM -- with the single
// substituted column patched on the fly.  HBM sees only the perm read and fully coalesced writes.
// Replaces varsens/saltelli.py:92-125 and :127-160.
//   flat row R = t*n + i:  t = 0: A_i | t = 1: B_i | t = 2+j: B_i with col j <- A_i[j]
//                          t = 2+k+j: A_i with col j <- B_i[j]
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
sample_flat_kernel(int k, int TI, SourceDev src, ScaleDev s, uint64_t i_lo, uint64_t i_hi, uint64_t row_begin,
                   uint64_t row_end, double *__restrict__ out) {
    extern __shared__ double smem[];
    double *A = smem;                       // [TI][k]
    double *B = smem + (size_t)TI * k;      // [TI][k]
    const uint64_t n = src.n;
    const uint64_t i0 = i_lo + (uint64_t)blockIdx.x * TI;
    const int rows = (int)((i0 + TI <= i_hi) ? TI : (i_hi - i0));
    const int cells = rows * k;
    for (int e = threadIdx.x; e < cells; e += blockDim.x) {
        int r = e / k, d = e - r * k;
        uint64_t i = i0 + r;
        A[e] = apply_scale(s, d, source_a(src, k, i, d));
        B[e] = apply_scale(s, d, source_b(src, k, src.perm[i], d));
    }
    __syncthreads();
    const int nblk = 2 + 2 * k;
    for (int t = 0; t < nblk; ++t) {
        uint64_t R0 = (uint64_t)t * n + i0;                 // first flat row of this run
        if (R0 + rows <= row_begin || R0 >= row_end) continue;
        const bool base_is_A = (t == 0) || (t >= 2 + k);
        const int j = (t < 2) ? -1 : (t < 2 + k ? t - 2 : t - 2 - k);
        const double *base = base_is_A ? A : B;
        const double *other = base_is_A ? B : A;
        int e_lo = (R0 < row_begin) ? (int)((row_begin - R0) * k) : 0;
        int e_hi = (R0 + rows > row_end) ? (int)((row_end - R0) * k) : cells;
        double *dst = out + (R0 - row_begin) * (uint64_t)k;  // may point before `out` when e_lo > 0; only [e_lo,e_hi) is touched
        for (int e = e_lo + threadIdx.x; e < e_hi; e += blockDim.x) {
            int d = e % k;
            double v = (d == j) ? other[e] : base[e];
            __stcs(dst + e, v);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// K3, bulk form (even k, 16-byte aligned output): persistent CTAs, warp-specialised.
//   14 warps    GENERATE the tile of TI = 32 base rows: A (M_1 rows) and B (shuffled M_2 rows), 2*TI*k radical inverses, into
//               one of two tile-buffer pairs -- the next tile is generated while the current one is being stored.  lane = row,
//               the warp walks one dimension at a time with the multiply-only digit loop of device.cuh (halton_pair): table
//               terms from shared memory for bases < 37, computed terms (double-double reciprocal) for the rest, so the
//               shared-memory table is 21 KB instead of 161 KB at k = 50.
//   1-2 warps   STORE the 2+2k flat blocks of the tile with the TMA: a block of the flat layout is the tile with ONE column
//               replaced, so the warp patches that column in place (lane = row: TI shared stores), issues one
//               cp.async.bulk.global.shared::cta of the whole TI*k-double tile (12.8 KB at k = 50), and restores the column
//               after the bulk read has drained; the A tile and the B tile alternate (N_j[j] is B with column j from A,
//               N_nj[j] is A with column j from B), so one bulk store is always in flight while the other tile is patched.
//               With two store warps (copies = 2) each owns its own copy of the tile pair and every second column.
// No thread touches the 171 GB going out: per flat block the SM issues ~70 instructions instead of ~40 per 8 bytes.
// Two addressings of the output: a window [row_begin,row_end) of Sample.flat() (mode 0: export batches), or the BASE-ROW
// shard [i_lo,i_hi) of every block (mode 1: out[(t*rows + i - i_lo)*k + c]; multi-GPU export: a rank generates only its rows).
// Measured (C4, k = 50, n = 2^22; tools/export_trace.py, profiles/r02_export_windows.txt): the serial part of a block in the
// store warp (wait for the buffer, patch, proxy fence, issue) takes 600-900 cycles, a 12.8 KB block at the HBM rate 590.
//   every block wanted (shard mode, windows longer than k blocks): ONE store warp with A/B alternation writes 7.0 TB/s; two
//     warps (four stores in flight per SM) only 6.2 TB/s -> copies = 1;
//   windows of at most k blocks (one family at a time, no alternation): one warp 4.0 TB/s, two warps 5.7 TB/s -> copies = 2.
// ---------------------------------------------------------------------------------------------
int launch_sample_flat(vs_ctx *c, int k, const SourceDev &src, const ScaleDev &s, uint64_t row_begin, uint64_t row_end, double *out);

struct ExportGeom {
    int k, TI, mode;
    int fast;                        // multiply-only digit loop + computed terms for the large bases (device.cuh: halton_pair)
    int copies;                      // copies of each tile (A, B): patched blocks of one family in flight at the same time
    uint64_t i_lo, i_hi;             // base rows covered by the launch
    uint64_t row_begin, row_end;     // mode 0: flat-row window
    int qb, qe;                      // ... its first and last flat row as (block, row in block): row_begin = qb n + rb,
    uint64_t rb, re;                 //     row_end - 1 = qe n + re
    uint32_t table_len;              // doubles of the term table copied to shared memory (0: read it from global memory)
    uint64_t ntiles;
    unsigned long long *trace;       // VS_TRACE: clock stamps of CTA 0's first EX_TRACE_TILES tiles ([tile][8]), else nullptr
};
constexpr int EX_TRACE_TILES = 48;
__device__ __forceinline__ void ex_stamp(const ExportGeom &g, uint64_t it, int slot, int lane) {
    if (g.trace && blockIdx.x == 0 && it < EX_TRACE_TILES && lane == 0) g.trace[it * 16 + slot] = clock64();
}

#ifndef EX_WAIT_HINT_NS
#define EX_WAIT_HINT_NS 500u   // short suspend hint of the mbarrier waits: the hand-over latency is on the tile's critical path
#endif
__device__ __forceinline__ void ex_bulk_store(double *dst, const double *src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void ex_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void ex_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void ex_fence_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

constexpr int EX_THREADS = 512, EX_STORE_WARPS = 2, EX_GEN = EX_THREADS - 32 * EX_STORE_WARPS;

__global__ void __launch_bounds__(EX_THREADS, 1)
sample_flat_bulk_kernel(ExportGeom g, SourceDev src, ScaleDev s, double *__restrict__ out) {
    extern __shared__ __align__(16) double smem[];
    const int k = g.k, TI = g.TI, NC = g.copies;
    // layout: bars[4] | generator prefix (device.cuh: halton_prefix) | tiles: per buffer pair (2): per copy (NC): A, B (TI*k each)
    // (the tiles are sources of cp.async.bulk: 16-byte aligned, as k is even and the table length is rounded up to even)
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem);                 // full[2], empty[2]
    const size_t tile = (size_t)TI * k;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        mbar_init(bars + 0, EX_GEN / 32);
        mbar_init(bars + 1, EX_GEN / 32);
        mbar_init(bars + 2, (uint32_t)NC);                   // every store warp releases the buffer pair
        mbar_init(bars + 3, (uint32_t)NC);
    }
    const HaltonPrefix gen = halton_prefix(smem + 4, k, src, s, g.table_len, g.fast != 0, g.fast == 1 ? EX_GEN / 32 : 0);
    const HaltonShared &hs = gen.hs;
    double *tiles = gen.table + ((g.table_len + 1) & ~1u);
    const double *T = g.table_len ? gen.table : src.h.terms;
    const uint64_t n = src.n;
    const uint64_t my_tiles = blockIdx.x < g.ntiles ? (g.ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if (warp >= EX_STORE_WARPS) {
        // ------------------------------------------ generators ------------------------------------------
        // lane = tile row, warp = a set of dimensions: all lanes of a warp walk the SAME base, so the digit loop has one trip
        // count per warp (no divergence), the base / magic / table row are warp-uniform, and the A chain (consecutive indices:
        // conflict-free table reads) and the B chain (permuted indices) of a row advance together as two independent chains.
        const int gw = warp - EX_STORE_WARPS;
        for (uint64_t it = 0; it < my_tiles; ++it) {
            const int pb = (int)(it & 1);
            const uint64_t i0 = g.i_lo + (blockIdx.x + it * gridDim.x) * (uint64_t)TI;
            const int rows = (int)((i0 + TI <= g.i_hi) ? TI : (g.i_hi - i0));
            double *A = tiles + (size_t)(2 * NC * pb) * tile, *B = A + tile;
            const bool live = lane < rows;
            const uint64_t i = i0 + (live ? lane : 0);
            if (gw == 1) ex_stamp(g, it, 0, lane);
            const uint64_t pi = src.perm[i];
            if (gw == 1 && pi != ~0ull) ex_stamp(g, it, 1, lane);                        // (the compare makes the stamp wait for the load)
            mbar_wait(bars + 2 + pb, (uint32_t)(((it >> 1) & 1) ^ 1), EX_WAIT_HINT_NS);   // the store warp is done with this buffer pair
            if (gw == 1) ex_stamp(g, it, 2, lane);
            auto emit = [&](int d, double pa, double pbv) {
                if (s.kind == VS_SCALE_LINEAR) {
                    pa = scale_value(VS_SCALE_LINEAR, gen.lb[d], gen.wr[d], pa);
                    pbv = scale_value(VS_SCALE_LINEAR, gen.lb[d], gen.wr[d], pbv);
                } else if (s.kind == VS_SCALE_POWER) {
                    pa = scale_value(VS_SCALE_POWER, gen.lb[d], gen.wr[d], pa);
                    pbv = scale_value(VS_SCALE_POWER, gen.lb[d], gen.wr[d], pbv);
                }
                if (live) {
                    A[(size_t)lane * k + d] = pa;
                    B[(size_t)lane * k + d] = pbv;
                    if (NC == 2) {
                        A[2 * tile + (size_t)lane * k + d] = pa;
                        B[2 * tile + (size_t)lane * k + d] = pbv;
                    }
                }
            };
            if (g.fast == 1) {
                // units of one table dimension or two computed-term dimensions, balanced over the generator warps (halton_schedule)
                const uint32_t ia[1] = {(uint32_t)(src.start + i)}, ib[1] = {(uint32_t)(src.start + n + pi)};
                halton_units<1>(gw, gen.ulist, k, ia, ib, hs, [&](int d, int, double pa, double pbv) { emit(d, pa, pbv); });
            } else if (g.fast == 2) {
                // comparison form (VS_EXPORT_SLOW_GEN=2): one dimension at a time, round-robin over the generator warps
                for (int d = gw; d < k; d += EX_GEN / 32) {
                    const uint32_t b = hs.base[d], ma = (uint32_t)(src.start + i), mb = (uint32_t)(src.start + n + pi);
                    double pa, pbv;
                    if (b == 2u) {
                        pa = (double)__brev(ma) * 2.3283064365386962890625e-10;
                        pbv = (double)__brev(mb) * 2.3283064365386962890625e-10;
                    } else {
                        const uint32_t ia[1] = {ma}, ib[1] = {mb};
                        double qa[1], qb[1];
                        if (d < HL_D0) halton_pair<true, 1>(ia, ib, b, hs.magic[d], hs.dl[d], hs.table_saddr + 8u * hs.off[d], nullptr, nullptr, qa, qb);
                        else halton_pair<false, 1>(ia, ib, b, hs.magic[d], hs.dl[d], 0u, hs.arh + (size_t)d * HL_J, hs.arl + (size_t)d * HL_J, qa, qb);
                        pa = qa[0];
                        pbv = qb[0];
                    }
                    emit(d, pa, pbv);
                }
            } else {
                for (int d = gw; d < k; d += EX_GEN / 32) {
                    double pa, pbv;
                    if (src.raw) {
                        pa = src.raw[i * (uint64_t)k + d];
                        pbv = src.raw[(n + pi) * (uint64_t)k + d];
                    } else {
                        const uint32_t b = hs.base[d];
                        const uint64_t magic = hs.magic[d];
                        uint32_t ma = (uint32_t)(src.start + i), mb = (uint32_t)(src.start + n + pi);
                        if (src.h.mode == VS_HALTON_HORNER) {
                            pa = radical_inverse_horner(b, magic, ma);
                            pbv = radical_inverse_horner(b, magic, mb);
                        } else if (b == 2u) {
                            pa = (double)__brev(ma) * 2.3283064365386962890625e-10;
                            pbv = (double)__brev(mb) * 2.3283064365386962890625e-10;
                        } else {
                            const double *row = T + hs.off[d];
                            pa = 0.0;
                            pbv = 0.0;
                            while ((ma | mb) != 0u) {                       // an exhausted index keeps adding row[0] == 0.0: exact
                                const uint32_t qa = (uint32_t)__umul64hi((uint64_t)ma, magic), qb = (uint32_t)__umul64hi((uint64_t)mb, magic);
                                pa = __dadd_rn(pa, row[ma - qa * b]);
                                pbv = __dadd_rn(pbv, row[mb - qb * b]);
                                row += b;
                                ma = qa;
                                mb = qb;
                            }
                        }
                    }
                    emit(d, pa, pbv);
                }
            }
            if (gw == 1) ex_stamp(g, it, 3, lane);
            ex_fence_async();                                   // my tile entries must be visible to the TMA (async proxy)
            __syncwarp();
            if (lane == 0) mbar_arrive(bars + pb);
            if (gw == 1) ex_stamp(g, it, 4, lane);
        }
        return;
    }
    // ---------------------------------------------- store warps ---------------------------------------------
    // Store warp c owns copy c of the tile pair (A_c, B_c) and the columns j = c mod NC: the serial part of a block -- wait for
    // the buffer's previous bulk read, restore + patch a column (32 shared stores), proxy fence, issue -- costs 600-900 cycles
    // of ONE warp (phase stamps, VS_TRACE), more than the 590 cycles a 12.8 KB block may take at the HBM rate; two warps
    // halve it.  Within a warp the A block and the B block of a column alternate, so one bulk store streams while the other
    // buffer is patched; a window that covers one family only still has one store in flight per warp.
    const int sw = warp;
    if (sw >= NC) return;
    const uint64_t shard = g.i_hi - g.i_lo;
    for (uint64_t it = 0; it < my_tiles; ++it) {
        const int pb = (int)(it & 1);
        const uint64_t i0 = g.i_lo + (blockIdx.x + it * gridDim.x) * (uint64_t)TI;
        const int rows = (int)((i0 + TI <= g.i_hi) ? TI : (g.i_hi - i0));
        double *A = tiles + (size_t)(2 * NC * pb + 2 * sw) * tile, *B = A + tile;        // this warp's copy
        mbar_wait(bars + pb, (uint32_t)((it >> 1) & 1), EX_WAIT_HINT_NS);
        if (sw == 0) ex_stamp(g, it, 5, lane);
        // blocks [t_min, t_max] of this tile intersect the window (R0(t) = t n + i0 is monotonic in t).  With the window ends
        // split on the host into (block, row) = (qb, rb) and (qe, re) no division is needed: block t covers the tile's rows
        // [i0, last] of that block, so t_min = qb if rb <= last else qb + 1, and t_max = qe if i0 <= re else qe - 1.  (The first
        // form divided two 64-bit numbers per tile: ~2k cycles of the store warp's 6k-cycle fixed cost per tile.)
        int t_min = 0, t_max = 2 * k + 1;
        if (g.mode == 0) {
            const uint64_t last = i0 + (uint64_t)rows - 1;
            t_min = g.rb <= last ? g.qb : g.qb + 1;
            t_max = i0 <= g.re ? g.qe : g.qe - 1;
        }
        auto wanted = [&](int t) { return t >= t_min && t <= t_max; };
        // one block of the flat layout: tile rows [r0, r1) that fall into the window, contiguous in HBM.  Only the first and
        // the last wanted block of a tile can be clipped; everything else is tile_dst + t * blk.  The descriptor is computed
        // BEFORE the wait for the buffer (the asm statements are ordering points for the compiler): the store warp's serial
        // work per block is what bounds the kernel (~560 cycles per 12.8 KB block, phase stamps), so nothing that can be done
        // early may sit between the wait and the bulk store.
        const uint64_t blk = (g.mode == 0 ? n : shard) * (uint64_t)k;                        // doubles per block of the output
        double *tile_dst = g.mode == 0 ? out + ((int64_t)i0 - (int64_t)g.row_begin) * (int64_t)k : out + (i0 - g.i_lo) * (uint64_t)k;
        auto describe = [&](int t, double *&dst, uint32_t &src_off, uint32_t &bytes) {
            int r0 = 0, r1 = rows;
            if (g.mode == 0 && (t == t_min || t == t_max)) {
                const uint64_t R0 = (uint64_t)t * n + i0;
                if (R0 < g.row_begin) r0 = (int)(g.row_begin - R0);
                if (R0 + rows > g.row_end) r1 = (int)(g.row_end - R0);
            }
            dst = tile_dst + (uint64_t)t * blk + (uint64_t)r0 * k;
            src_off = (uint32_t)r0 * (uint32_t)k;
            bytes = (uint32_t)((r1 - r0) * k * 8);
        };
        // Every bulk store is its own group; groups drain in order.  A buffer may be patched again once ITS last group has
        // been read out of shared memory: if the newest group belongs to the other buffer, "all but one group done" is enough
        // (that one keeps streaming while this buffer is patched), else everything has to be done.
        int lastbuf = -1;                                       // buffer of the newest group: 0 = A, 1 = B
        int cA = -1, cB = -1;                                   // column currently patched in A / B
        double vA = 0.0, vB = 0.0;                              // ... and its original value (this lane's row)
        auto issue = [&](int t, double *buf, int which, int &pcol, double &pval, int col, double orig, double repl) {
            double *dst;
            uint32_t src_off, bytes;
            describe(t, dst, src_off, bytes);
            if (lane == 0) {
                if (lastbuf == which) ex_wait_read<0>();
                else ex_wait_read<1>();
            }
            __syncwarp();
            if (col >= 0) {
                if (lane < rows) {
                    if (pcol >= 0) buf[(size_t)lane * k + pcol] = pval;
                    buf[(size_t)lane * k + col] = repl;
                }
                pcol = col;
                pval = orig;
                ex_fence_async();
                __syncwarp();
            }
            if (lane == 0) {
                ex_bulk_store(dst, buf + src_off, bytes);
                ex_commit();
            }
            lastbuf = which;
        };
        if (sw == 0 && wanted(1)) issue(1, B, 1, cB, vB, -1, 0.0, 0.0);             // M_2
        if (sw == NC - 1 && wanted(0)) issue(0, A, 0, cA, vA, -1, 0.0, 0.0);        // M_1
        // columns j with a wanted block: N_j[j] is block 2 + j, N_nj[j] is block 2 + k + j
        const int jb_lo = max(t_min - 2, 0), jb_hi = min(t_max - 2, k - 1);                 // N_j
        const int ja_lo = max(t_min - 2 - k, 0), ja_hi = min(t_max - 2 - k, k - 1);         // N_nj
        int j_lo = jb_lo <= jb_hi ? (ja_lo <= ja_hi ? min(jb_lo, ja_lo) : jb_lo) : ja_lo;
        const int j_hi = jb_lo <= jb_hi ? (ja_lo <= ja_hi ? max(jb_hi, ja_hi) : jb_hi) : ja_hi;
        j_lo += (sw - j_lo % NC + NC) % NC;                     // first column >= j_lo with j = sw mod NC
        for (int j = j_lo; j <= j_hi; j += NC) {
            const bool nb = j >= jb_lo && j <= jb_hi, na = j >= ja_lo && j <= ja_hi;
            if (!nb && !na) continue;
            // column j is unpatched in this copy (its patched columns are < j)
            const double a_j = lane < rows ? A[(size_t)lane * k + j] : 0.0;
            const double b_j = lane < rows ? B[(size_t)lane * k + j] : 0.0;
            if (nb) issue(2 + j, B, 1, cB, vB, j, b_j, a_j);                        // N_j[j] = B with column j from A
            if (na) issue(2 + k + j, A, 0, cA, vA, j, a_j, b_j);                    // N_nj[j] = A with column j from B
        }
        if (sw == 0) ex_stamp(g, it, 6, lane);
        if (lane == 0) ex_wait_read<0>();                       // this warp's tile buffers may be overwritten by the generators now
        __syncwarp();
        if (lane == 0) mbar_arrive(bars + 2 + pb);
        if (sw == 0) ex_stamp(g, it, 7, lane);
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // all bulk stores complete before the CTA exits
}

// base rows touched by a flat-row window: if it lies inside one block, that block's row range; else all of them
static void window_rows(uint64_t n, uint64_t row_begin, uint64_t row_end, uint64_t *i_lo, uint64_t *i_hi) {
    *i_lo = 0;
    *i_hi = n;
    const uint64_t t_first = row_begin / n, t_last = (row_end - 1) / n;
    if (t_first == t_last) {
        *i_lo = row_begin - t_first * n;
        *i_hi = row_end - t_first * n;
    } else if (t_last == t_first + 1 && row_end - t_last * n <= row_begin - t_first * n) {
        // two arcs that do not overlap: [row_begin - t_first n, n) of the first block and [0, row_end - t_last n) of the next.
        // (kept simple: generate everything; the arcs case only matters for windows shorter than one block)
    }
}

static int launch_sample_flat_bulk(vs_ctx *c, int k, const SourceDev &src, const ScaleDev &s, int mode, uint64_t i_lo, uint64_t i_hi,
                                   uint64_t row_begin, uint64_t row_end, double *out, bool *done) {
    *done = false;
    if ((k & 1) || (reinterpret_cast<uintptr_t>(out) & 15) || i_hi <= i_lo) return VS_OK;
    ExportGeom g{};
    g.k = k;
    g.mode = mode;
    g.i_lo = i_lo;
    g.i_hi = i_hi;
    g.row_begin = row_begin;
    g.row_end = row_end;
    if (mode == 0) {
        g.qb = (int)(row_begin / src.n);
        g.rb = row_begin % src.n;
        g.qe = (int)((row_end - 1) / src.n);
        g.re = (row_end - 1) % src.n;
    }
    const size_t avail = c->smem_optin;
    const size_t fixed = (4 + halton_prefix_doubles(k) + 2) * sizeof(double);      // mbarriers, generator prefix without the table
    // fast generator: table rows only for the small bases (dimensions < HL_D0), computed terms for the rest
    g.fast = (!src.raw && src.h.mode != VS_HALTON_HORNER && src.h.arith_ok && c->opt.export_slow_gen != 1) ? (c->opt.export_slow_gen == 2 ? 2 : 1) : 0;
    const size_t tab_terms = src.raw ? 0 : g.fast ? halton_table_prefix(c->halton) : src.h.total_terms;
    const size_t tab = ((tab_terms + 1) & ~(size_t)1) * sizeof(double);
    // tile height: 32 rows (one lane per row in the store warp); two copies of every tile if they fit beside the term table
    // store warps / tile copies: one when A and B blocks of the same column alternate (every block wanted), else two (see above)
    int TI = 32, copies = (mode == 1 || g.qe - g.qb >= k) ? 1 : 2;
    if (c->opt.export_copies == 1 || c->opt.export_copies == 2) copies = c->opt.export_copies;   // VS_EXPORT_COPIES
    bool with_table = !src.raw && src.h.mode != VS_HALTON_HORNER && fixed + tab + 4 * (size_t)TI * k * 8 <= avail;
    if (g.fast && (!with_table || halton_unit_count(k) > HL_MAX_UNITS)) g.fast = 0;   // (k beyond ~440: generic loop, table in global memory)
    if (!with_table)
        while (TI > 1 && fixed + 4 * (size_t)TI * k * 8 > avail) TI >>= 1;
    if (fixed + (with_table ? tab : 0) + 4 * (size_t)copies * TI * k * 8 > avail) copies = 1;
    if (fixed + (with_table ? tab : 0) + 4 * (size_t)copies * TI * k * 8 > avail) return VS_OK;
    if (((size_t)TI * k * 8) >= (1u << 20)) return VS_OK;                       // bulk copy size field
    g.TI = TI;
    g.copies = copies;
    g.table_len = with_table ? (uint32_t)tab_terms : 0;
    g.ntiles = (i_hi - i_lo + TI - 1) / TI;
    size_t smem = fixed + (with_table ? tab : 0) + 4 * (size_t)copies * TI * k * 8;
    if (smem > avail) smem = avail;
    static size_t smem_set[64] = {};
    if (c->device >= 64 || smem_set[c->device] < smem) {
        VS_CUDA(cudaFuncSetAttribute(sample_flat_bulk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        if (c->device < 64) smem_set[c->device] = smem;
    }
    const unsigned grid = (unsigned)(g.ntiles < (uint64_t)c->sm_count ? g.ntiles : (uint64_t)c->sm_count);
    g.trace = nullptr;
    if (!c->opt.trace.empty()) {
        VS_CUDA(cudaMalloc(&g.trace, EX_TRACE_TILES * 16 * sizeof(unsigned long long)));
        VS_CUDA(cudaMemsetAsync(g.trace, 0, EX_TRACE_TILES * 16 * sizeof(unsigned long long), c->stream));
    }
    time_begin(c);
    sample_flat_bulk_kernel<<<grid, EX_THREADS, smem, c->stream>>>(g, src, s, out);
    time_end(c);
    c->launches++;
    VS_CUDA(cudaGetLastError());
    if (g.trace) {
        // CTA 0, per tile: generator warp 1: loop top, perm loaded, buffer free, tile generated, arrived | store warp: tile
        // full, stores issued, buffer released -- cycles relative to the first stamp
        std::vector<unsigned long long> h(EX_TRACE_TILES * 16);
        VS_CUDA(cudaStreamSynchronize(c->stream));
        VS_CUDA(cudaMemcpy(h.data(), g.trace, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        VS_CUDA(cudaFree(g.trace));
        if (FILE *f = fopen(c->opt.trace.c_str(), "a")) {
            fprintf(f, "# sample_flat_bulk_kernel k=%d TI=%d copies=%d fast=%d mode=%d tiles/CTA=%llu: tile | gen: top perm free done arrived | store: full issued released\n",
                    k, g.TI, g.copies, g.fast, mode, (unsigned long long)((g.ntiles + grid - 1) / grid));
            for (int t = 0; t < EX_TRACE_TILES && h[t * 16]; ++t) {
                fprintf(f, "%3d |", t);
                for (int q = 0; q < 8; ++q) fprintf(f, " %8lld%s", (long long)(h[t * 16 + q] - h[0]), q == 4 ? " |" : "");
                fprintf(f, " | dims of generator warp 1 done at:");
                for (int q = 8; q < 16 && h[t * 16 + q]; ++q) fprintf(f, " %8lld", (long long)(h[t * 16 + q] - h[0]));
                fprintf(f, "\n");
            }
            fclose(f);
        }
    }
    *done = true;
    return VS_OK;
}

// Base-row shard of every block (vs_sample_flat_shard): out[(t*rows + i - i_begin)*k + c], rows = i_end - i_begin.
int launch_sample_shard(vs_ctx *c, int k, const SourceDev &src, const ScaleDev &s, uint64_t i_begin, uint64_t i_end, double *out) {
    if (i_end <= i_begin) return VS_OK;
    bool done = false;
    VS_TRY(launch_sample_flat_bulk(c, k, src, s, 1, i_begin, i_end, 0, 0, out, &done));
    if (done) return VS_OK;
    // odd k / unaligned output: block by block through the scalar kernel (each block's shard rows are one flat-row window)
    const uint64_t rows = i_end - i_begin;
    for (int t = 0; t < 2 + 2 * k; ++t)
        VS_TRY(launch_sample_flat(c, k, src, s, (uint64_t)t * src.n + i_begin, (uint64_t)t * src.n + i_end, out + (uint64_t)t * rows * k));
    return VS_OK;
}

int launch_sample_flat(vs_ctx *c, int k, const SourceDev &src, const ScaleDev &s, uint64_t row_begin, uint64_t row_end,
                       double *out) {
    if (row_end <= row_begin) return VS_OK;
    const uint64_t n = src.n;
    if (!c->opt.no_bulk_export) {
        uint64_t bl, bh;
        window_rows(n, row_begin, row_end, &bl, &bh);
        bool done = false;
        VS_TRY(launch_sample_flat_bulk(c, k, src, s, 0, bl, bh, row_begin, row_end, out, &done));
        if (done) return VS_OK;
    }
    // base rows touched by the window: if it spans a whole block, all of them; else the union of <= 2 arcs.
    uint64_t i_lo = 0, i_hi = n;
    uint64_t t_first = row_begin / n, t_last = (row_end - 1) / n;
    if (t_first == t_last) {
        i_lo = row_begin - t_first * n;
        i_hi = row_end - t_first * n;
    }
    // TI rows per CTA: as many as fit ~48 KB of shared memory, at most 32.
    size_t per_row = 2 * (size_t)k * sizeof(double);
    int TI = (int)(48 * 1024 / per_row);
    if (TI > 32) TI = 32;
    if (TI < 1) {
        TI = 1;
        VS_REQUIRE(per_row <= c->smem_optin, VS_ERR_UNSUPPORTED, "k=%d needs %zu bytes of shared memory per row", k, per_row);
    }
    size_t smem = per_row * TI;
    if (smem > 48 * 1024) VS_CUDA(cudaFuncSetAttribute(sample_flat_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    uint64_t tiles = (i_hi - i_lo + TI - 1) / TI;
    VS_REQUIRE(tiles < (1ull << 31), VS_ERR_RANGE, "too many tiles");
    time_begin(c);
    sample_flat_kernel<<<(unsigned)tiles, 256, smem, c->stream>>>(k, TI, src, s, i_lo, i_hi, row_begin, row_end, out);
    time_end(c);
    c->launches++;
    VS_CUDA(cudaGetLastError());
    return VS_OK;
}

}  // namespace vs
