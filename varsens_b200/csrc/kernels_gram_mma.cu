// Estimator reductions on given values, tensor path.
//
// Computes the same partial-sum vector as gram_kernel (kernels_vals.cu) -- the symmetric Gram
// G = sum_i v_i v_i^T of the per-row vector v_i = (f(M_1[i]), f(M_2[i]), f(N_j[.][i]), f(N_nj[.][i])) plus the
// shifted sums for var_y, i.e. everything varsens/saltelli.py:577-622 reads -- but shaped for the hardware:
//
//   * the value layout handed over by the reference API is column-major already (flat() order: all rows of M_1,
//     then M_2, ... -> fvals[t * rows + r]), so a chunk of RC rows is m contiguous runs of RC doubles.  One producer
//     warp moves them with 1-D bulk copies (cp.async.bulk, completion on an mbarrier) into a ring of shared-memory
//     stages Yt[p][RC + 4]; nothing is transposed and no thread waits on a global load.
//   * consumer warps run the Gram update on the FP64 tensor path (mma.sync m8n8k4): the fragment
//     Yt[8P + lane/4][r0 + lane%4] is both the A and the B operand of G[P][Q] += Y[r0..r0+4, P]^T Y[r0..r0+4, Q]
//     and loads conflict-free (pitch = 4 mod 16).  A warp owns one ST x ST super-tile of 8x8 blocks (its accumulators
//     never leave registers) and a subset of the 4-row steps of every chunk.
//   * row subsets, then CTAs, are combined in a fixed order -> bit-reproducible.
//   * GEN form (l > 1 outputs, or an odd row count): block t of the value layout is a contiguous run of rows*l doubles
//     fvals[(t*rows + r)*l + o], so a chunk of RC rows of block t is still ONE bulk copy of RC*l doubles into
//     Yt[t][mis_t + r*l + o]; mis_t = 1 when the run starts 8 bytes off a 16-byte boundary (rows*l odd, t odd): the copy
//     then starts one element early and is rounded up to 16 bytes (the neighbours it touches belong to the same
//     array).  Coordinate c = t*l + o (the order of the partial-sum vector); each lane keeps the shared-memory offset of
//     its coordinate of every block of its super-tile in registers, padded coordinates point at a zero row.
//
// Bound: max(HBM, FP64).  k = 20: 336 B and 21 DMMA (10.8 kflop) per row -> 0.22 ms of HBM and 0.30 ms of FP64 for
// n = 2^22 on a B200.
#include "device.cuh"
#include "vs_internal.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <type_traits>
#include <vector>

namespace vs {

struct MmaGeom {
    int m, nb, mpad;       // coordinates, 8-wide blocks, padded coordinates
    int l, nt;             // outputs per evaluation, value blocks (2 + 2k); m = nt * l
    int gen;               // GEN form (l > 1 or odd rows*l): per-lane coordinate offsets, see the header
    int oddrun;            // rows * l is odd: the runs of odd blocks start 8 bytes off a 16-byte boundary
    int imax;              // block rows that are needed (nb, or 1 without the second-order block)
    int nsb, nunits;       // super-blocks per side, super-tiles in use
    int upc, passes;       // super-tiles per CTA, grid.y
    int rs, warps;         // row subsets per super-tile, consumer warps per CTA
    int rc, pitch, nstage; // rows per chunk, doubles per staged column, ring depth
    int second;
    int sumu;              // position of super-tile (0,0) in the list: its warps also accumulate the shifted sums
    unsigned char witem[32];   // consumer warp -> work item (super-tile of this pass * rs + row subset), 255 = idle
    unsigned char ui[128], uj[128];   // super-tile list, heaviest first
    int debug;             // elimination experiments (VS_GRAM_DEBUG): 1 = no Gram update, 2 = no copies
};

// global -> shared bulk copy (16-byte aligned on both sides, size a multiple of 16), completion counted on `bar`
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}


// The 4-row steps `rsub, rsub + rs, ...` of one staged chunk for the super-tile whose first blocks are (bi0, bj0).
//   DIAG : row and column operands are the same blocks (only x <= y is needed, and the fragments are shared when `share`).
//   GUARD: some of the ST x ST blocks may not exist (edge super-tiles, first-order-only mode) -> uniform predicates.
//   FULL : every row of the chunk is valid (all chunks but the last one) -> no per-lane row predicate.
// Keep this loop lean: it issues next to the DMMAs (a first version that re-derived `valid` from the kernel arguments for
// every predicated load ran 376 instructions per step and was issue-bound at 0.89 ms; see profiles/r01_gram_mma_ncu.txt).
//   GEN  : l > 1 or odd rows: the fragment of block x is at Ya[offa[x] + r0 * l] (offa, offb: per-lane register tables) and
//          the shifted sums cover the coordinates c < 2l of the diagonal super-tile (sS, sQ: one pair per block).
template <int ST, bool DIAG, bool GUARD, bool FULL, bool GEN>
__device__ __forceinline__ void mma_steps(double (&acc)[ST * ST][2], double (&sS)[GEN ? ST : 1], double (&sQ)[GEN ? ST : 1],
                                          const double *__restrict__ Ya, const double *__restrict__ Yb, int colstride, int valid,
                                          int rsub, int rs, int lane, int xmax, int ymax, int share, bool do_sums,
                                          const double (&shiftv)[GEN ? ST : 1], const int (&offa)[GEN ? ST : 1],
                                          const int (&offb)[GEN ? ST : 1], int l, unsigned summask) {
    const int ksteps = (valid + 3) >> 2;
    const int lrow = lane & 3;
#pragma unroll 1
    for (int ks = rsub; ks < ksteps; ks += rs) {
        const int r0 = GEN ? (ks << 2) * l : (ks << 2);          // element offset of the step's first row inside a run
        const bool rv = FULL || ((ks << 2) + lrow < valid);
        double fa[ST], fb[ST];
#pragma unroll
        for (int x = 0; x < ST; ++x) {
            const bool on = (!GUARD || x < xmax) && rv;
            fa[x] = 0.0;
            if (on) fa[x] = GEN ? Ya[offa[x] + r0] : Ya[x * colstride + r0];
        }
        if (DIAG && (!GUARD || share)) {
#pragma unroll
            for (int y = 0; y < ST; ++y) fb[y] = fa[y];
        } else {
            // (without the second-order block only block row 0 is loaded on the row side; the column side needs them all)
#pragma unroll
            for (int y = 0; y < ST; ++y) {
                const bool on = (!GUARD || y < ymax) && rv;
                fb[y] = 0.0;
                if (on) fb[y] = GEN ? Yb[offb[y] + r0] : Yb[y * colstride + r0];
            }
        }
        if (DIAG && do_sums) {
            if constexpr (!GEN) {
                const double d = rv ? fa[0] - shiftv[0] : 0.0;      // lanes 0-3: f(M_1) rows, lanes 4-7: f(M_2) rows
                sS[0] += d;
                sQ[0] = fma(d, d, sQ[0]);
            } else {
#pragma unroll
                for (int x = 0; x < ST; ++x)
                    if (summask >> x & 1u) {                         // this lane's coordinate of block x is one of the 2l summed ones
                        const double d = rv ? fa[x] - shiftv[x] : 0.0;
                        sS[x] += d;
                        sQ[x] = fma(d, d, sQ[x]);
                    }
            }
        }
#pragma unroll
        for (int x = 0; x < ST; ++x)
#pragma unroll
            for (int y = DIAG ? x : 0; y < ST; ++y)
                if (!GUARD || (x < xmax && y < ymax)) dmma_m8n8k4(acc[x * ST + y][0], acc[x * ST + y][1], fa[x], fb[y]);
    }
}

constexpr int MMA_BAR_DOUBLES = 16;     // full[8] + empty[8]
constexpr int MMA_MAX_STAGES = 8;

// MULTI: several super-tiles (ST = 4 or 2); otherwise one diagonal super-tile.  The 2 x 2 form needs <= 64 registers, so a CTA
// may hold 31 consumer warps: 28 super-tiles at k = 50 fit ONE pass over the data (15 warps needed two: 6.85 GB of DRAM reads
// for 3.42 GB of values, ncu) and light configurations get three row subsets per super-tile.
template <int ST, bool MULTI, bool GUARD, bool GEN>
__global__ void __launch_bounds__(MULTI ? (ST == 2 ? 1024 : 512) : 384)
gram_mma_kernel(MmaGeom g, uint64_t rows, const double *__restrict__ fvals, const double *__restrict__ shift,
                double *__restrict__ blockpart) {
    extern __shared__ __align__(16) double smem[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem);
    uint64_t *empty = full + MMA_MAX_STAGES;
    double *stages = smem + MMA_BAR_DOUBLES;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int W = g.warps;
    // staged rows per stage: the mpad padded coordinates, or (GEN) the nt value blocks plus one zero row for the padding
    const int stage_rows = GEN ? g.nt + 1 : g.mpad;
    const int stage_elems = stage_rows * g.pitch;

    if (threadIdx.x == 0) {
        for (int s = 0; s < g.nstage; ++s) {
            mbar_init(full + s, 1);
            mbar_init(empty + s, (uint32_t)W);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // the padded coordinates m .. mpad-1 (GEN: the zero row) are never copied: zero them once
    const int zrow0 = GEN ? g.nt : g.m, zrows = stage_rows - zrow0;
    for (int e = threadIdx.x; e < g.nstage * zrows * g.pitch; e += blockDim.x) {
        const int s = e / (zrows * g.pitch), rem = e - s * (zrows * g.pitch);
        stages[(size_t)s * stage_elems + (size_t)zrow0 * g.pitch + rem] = 0.0;
    }
    __syncthreads();

    const uint32_t nchunks = (uint32_t)((rows + g.rc - 1) / g.rc);                 // rows < 2^36 (checked on the host)
    const uint32_t cnt = blockIdx.x < nchunks ? (nchunks - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int last_valid = (int)(rows - (uint64_t)(nchunks - 1) * g.rc);          // rows of the last chunk

    double acc[ST * ST][2];
#pragma unroll
    for (int t = 0; t < ST * ST; ++t) { acc[t][0] = 0.0; acc[t][1] = 0.0; }
    constexpr int NS = GEN ? ST : 1;
    double sS[NS], sQ[NS];
#pragma unroll
    for (int x = 0; x < NS; ++x) { sS[x] = 0.0; sQ[x] = 0.0; }

    // work item of this warp: the host spreads the super-tiles over the four sub-partitions by DMMA count (the FP64 pipe is
    // per sub-partition, and a diagonal or edge super-tile has far fewer 8x8 tiles than an interior one)
    const int item = warp < W ? g.witem[warp] : 255;
    const int ul = item == 255 ? 0 : item / g.rs, rsub = item == 255 ? 0 : item - ul * g.rs;
    const int u = blockIdx.y * g.upc + ul;
    const bool active = item != 255 && u < g.nunits;
    const int I = active ? g.ui[u] : 0, J = active ? g.uj[u] : 0;

    if (warp == W) {
        // ------------------------------------ producer ------------------------------------
        int s = 0;
        uint32_t par = 0;
        uint32_t ch = blockIdx.x;
        for (uint32_t c = 0; c < cnt; ++c, ch += gridDim.x) {
            mbar_wait(empty + s, par ^ 1u, MBAR_HINT_NS);
            const uint64_t r0 = (uint64_t)ch * g.rc;
            const uint32_t valid = ch + 1 == nchunks ? (uint32_t)last_valid : (uint32_t)g.rc;
            // One elected lane issues every copy from a warp-uniform loop: the operands stay in uniform registers.  (A
            // lane-strided loop compiles to an ELECT + 5x R2UR + UBLKCP round per lane, ~100 cycles per copy, and the
            // producer became the bottleneck: 0.89 ms instead of the 0.3 ms FP64 bound at k = 20, n = 2^22.)
            if (g.debug == 2) {
                if (lane == 0) mbar_arrive(full + s);
            } else if (elect_one()) {
                double *dst = stages + (size_t)s * stage_elems;
                if constexpr (!GEN) {
                    mbar_arrive_expect_tx(full + s, (uint32_t)g.m * valid * 8u);
                    const double *src = fvals + r0;
#pragma unroll 4
                    for (int t = 0; t < g.m; ++t) bulk_g2s(dst + (size_t)t * g.pitch, src + (uint64_t)t * rows, valid * 8u, full + s);
                } else {
                    // run of block t: valid*l doubles from fvals[(t*rows + r0)*l]; even blocks start on a 16-byte boundary, odd
                    // blocks too unless rows*l is odd -- then they start one element early.  Sizes rounded up to 16 bytes.
                    const uint32_t nel = valid * (uint32_t)g.l;
                    const uint32_t be = ((nel + 1u) & ~1u) * 8u, bo = ((nel + (uint32_t)g.oddrun + 1u) & ~1u) * 8u;
                    mbar_arrive_expect_tx(full + s, (uint32_t)(g.nt / 2) * (be + bo));
                    const double *src = fvals + r0 * (uint64_t)g.l;
                    const uint64_t run = rows * (uint64_t)g.l;
#pragma unroll 2
                    for (int t = 0; t < g.nt; t += 2) {
                        bulk_g2s(dst + (size_t)t * g.pitch, src + (uint64_t)t * run, be, full + s);
                        bulk_g2s(dst + (size_t)(t + 1) * g.pitch, src + (uint64_t)(t + 1) * run - g.oddrun, bo, full + s);
                    }
                }
            }
            __syncwarp();
            if (++s == g.nstage) { s = 0; par ^= 1u; }
        }
    } else if (warp < W) {
        // ------------------------------------ consumers -----------------------------------
        const int foff = (lane >> 2) * g.pitch + (lane & 3);
        const bool do_sums = active && u == g.sumu;
        const int colstride = 8 * g.pitch;
        const int xmax = g.imax - ST * I, ymax = g.nb - ST * J;   // blocks of this super-tile that exist (row / column side)
        const double *Ya0 = stages + (GEN ? 0 : foff + (ST * I) * colstride), *Yb0 = stages + (GEN ? 0 : foff + (ST * J) * colstride);
        // GEN: shared-memory offset of this lane's coordinate c = 8*block + lane/4 at row lane%4 of a chunk, for every block of
        // the super-tile: value block t = c / l (row t of the stage, shifted by one element when its run is misaligned),
        // output o = c % l, row stride l.  Coordinates >= m read the zero row.
        int offa[NS], offb[NS];
        double shiftv[NS];
        unsigned summask = 0;
#pragma unroll
        for (int x = 0; x < NS; ++x) { offa[x] = 0; offb[x] = 0; shiftv[x] = 0.0; }
        if constexpr (GEN) {
            auto off_of = [&](int c) {
                if (c >= g.m) return g.nt * g.pitch + (lane & 3) * g.l;
                const int t = c / g.l, o = c - t * g.l;
                return t * g.pitch + ((t & 1) ? g.oddrun : 0) + o + (lane & 3) * g.l;
            };
#pragma unroll
            for (int x = 0; x < ST; ++x) {
                const int ca = 8 * (ST * I + x) + (lane >> 2), cb = 8 * (ST * J + x) + (lane >> 2);
                offa[x] = off_of(ca);
                offb[x] = off_of(cb);
                if (do_sums && ca < 2 * g.l) {
                    summask |= 1u << x;
                    shiftv[x] = shift ? shift[ca % g.l] : 0.0;
                }
            }
        } else {
            shiftv[0] = shift ? *shift : 0.0;
        }
        int s = 0;
        uint32_t par = 0;
        uint32_t ch = blockIdx.x;
        for (uint32_t c = 0; c < cnt; ++c, ch += gridDim.x) {
            mbar_wait(full + s, par, MBAR_HINT_NS);
            if (active && g.debug != 1) {
                const double *Ya = Ya0 + (size_t)s * stage_elems, *Yb = Yb0 + (size_t)s * stage_elems;
                const bool fullc = ch + 1 != nchunks || last_valid == g.rc;
                auto run = [&](auto diag, auto guard) {
                    constexpr bool D = decltype(diag)::value, G = decltype(guard)::value;
                    if (fullc) mma_steps<ST, D, G, true, GEN>(acc, sS, sQ, Ya, Yb, colstride, g.rc, rsub, g.rs, lane, xmax, ymax, g.second, D && do_sums, shiftv, offa, offb, g.l, summask);
                    else mma_steps<ST, D, G, false, GEN>(acc, sS, sQ, Ya, Yb, colstride, last_valid, rsub, g.rs, lane, xmax, ymax, g.second, D && do_sums, shiftv, offa, offb, g.l, summask);
                };
                using T_ = std::true_type;
                using F_ = std::false_type;
                if constexpr (!MULTI) {
                    run(T_{}, std::integral_constant<bool, GUARD>{});
                } else {
                    const bool interior = g.second && xmax >= ST && ymax >= ST;      // every block of the super-tile exists
                    if (I == J) { if (interior) run(T_{}, F_{}); else run(T_{}, T_{}); }
                    else { if (interior) run(F_{}, F_{}); else run(F_{}, T_{}); }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(empty + s);
            if (++s == g.nstage) { s = 0; par ^= 1u; }
        }
    }

    // ---- combine the row subsets of every super-tile in subset order (every copy has landed: all full barriers were waited on) ----
    __syncthreads();
    constexpr int SD = 8 * ST;                                  // super-tile side in coordinates
    double *img = stages;                                       // [upc][SD][SD]
    double *sums = img + (size_t)g.upc * SD * SD;               // [rs][NS][32][2]: (block, lane) = (coordinate, row mod 4)
    for (int round = 0; round < g.rs; ++round) {
        if (active && rsub == round) {
            double *mine = img + (size_t)ul * SD * SD;
#pragma unroll
            for (int x = 0; x < ST; ++x)
#pragma unroll
                for (int y = 0; y < ST; ++y) {
                    const int row = 8 * x + (lane >> 2), col = 8 * y + 2 * (lane & 3);   // C fragment: (lane/4, 2*(lane%4)+{0,1})
                    double *dst = mine + row * SD + col;
                    if (round == 0) { dst[0] = acc[x * ST + y][0]; dst[1] = acc[x * ST + y][1]; }
                    else { dst[0] += acc[x * ST + y][0]; dst[1] += acc[x * ST + y][1]; }
                }
            if (u == g.sumu) {
#pragma unroll
                for (int x = 0; x < NS; ++x) {
                    sums[((round * NS + x) * 32 + lane) * 2 + 0] = sS[x];
                    sums[((round * NS + x) * 32 + lane) * 2 + 1] = sQ[x];
                }
            }
        }
        __syncthreads();
    }
    const size_t per_block = (size_t)g.mpad * g.mpad + 4 * (size_t)g.l;
    double *bp = blockpart + (size_t)blockIdx.x * per_block;
    for (int q = 0; q < g.upc; ++q) {
        const int uq = blockIdx.y * g.upc + q;
        if (uq >= g.nunits) break;
        const int Iq = g.ui[uq], Jq = g.uj[uq];
        for (int e = threadIdx.x; e < SD * SD; e += blockDim.x) {
            const int row = e / SD, col = e - row * SD;
            const int gp = SD * Iq + row, gq = SD * Jq + col;
            if (gp < g.mpad && gq < g.mpad) bp[(size_t)gp * g.mpad + gq] = img[(size_t)q * SD * SD + e];
        }
    }
    if ((int)blockIdx.y == g.sumu / g.upc && (int)threadIdx.x < 4 * g.l) {
        // S_A[l], S_B[l], Q_A[l], Q_B[l] (coordinate c = t*l + o, t in {0, 1}): subsets in order, the four row lanes in order
        const int c = threadIdx.x % (2 * g.l), which = threadIdx.x / (2 * g.l);
        const int x = GEN ? c >> 3 : 0, cl = c & 7;
        double s = 0.0;
        for (int round = 0; round < g.rs; ++round)
            for (int ln = 0; ln < 4; ++ln) s += sums[((round * NS + x) * 32 + cl * 4 + ln) * 2 + which];
        bp[(size_t)g.mpad * g.mpad + threadIdx.x] = s;
    }
}

// per-CTA dense images (mpad x mpad + 4l sums) -> packed partial-sum vector; entries that were not computed are 0.
// One warp per entry: lane l adds CTAs l, l+32, ... in order, then a fixed shuffle tree (reproducible for a given grid).
__global__ void __launch_bounds__(256) gram_mma_scatter_kernel(int m, int mpad, int l, int pmax, int nblocks, const double *__restrict__ blockpart,
                                                               double *__restrict__ partials) {
    const size_t per_block = (size_t)mpad * mpad + 4 * (size_t)l;
    const int lane = threadIdx.x & 31;
    const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nent = (long long)m * (m + 1) / 2;
    if (w >= nent + 4 * l) return;
    const double *src;
    long long dst;
    bool computed = true;
    if (w < 4 * l) {
        src = blockpart + (size_t)mpad * mpad + w;
        dst = w;
    } else {
        long long rem = w - 4 * l;
        int p = 0, rowlen = m;
        while (rem >= rowlen) { rem -= rowlen; --rowlen; ++p; }
        const int q = p + (int)rem;
        src = blockpart + (size_t)p * mpad + q;
        dst = w;
        computed = p < pmax;
    }
    double s = 0.0;
    if (computed)
        for (int b = lane; b < nblocks; b += 32) s += src[(size_t)b * per_block];
    s = warp_sum(s);
    if (lane == 0) partials[dst] = s;
}

template <int ST, bool MULTI, bool GUARD, bool GEN>
static int launch_mma_t(vs_ctx *c, const MmaGeom &g, size_t smem, uint64_t rows, const double *fvals, const double *shift_dev,
                        double *partials) {
    auto kern = gram_mma_kernel<ST, MULTI, GUARD, GEN>;
    VS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int threads = (g.warps + 1) * 32;
    int occ = 1;
    VS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem));
    if (occ < 1) occ = 1;
    if (occ > 2) occ = 2;
    const uint64_t nchunks = (rows + g.rc - 1) / g.rc;
    int gx = (int)(nchunks < (uint64_t)occ * c->sm_count ? nchunks : (uint64_t)occ * c->sm_count);
    if (gx < 1) gx = 1;
    const size_t per_block = (size_t)g.mpad * g.mpad + 4 * (size_t)g.l;
    VS_TRY(ensure(c, c->block_buf, (size_t)gx * per_block * sizeof(double)));
    time_begin(c);
    kern<<<dim3(gx, g.passes), threads, smem, c->stream>>>(g, rows, fvals, shift_dev, (double *)c->block_buf.p);
    time_end(c);
    c->launches++;
    VS_CUDA(cudaGetLastError());
    if (!c->opt.trace.empty()) {
        // VS_TRACE: the instantiation and plan that ran (the tests read chunks per CTA = ceil(ceil(rows / rc) / gx) from it)
        if (FILE *f = fopen(c->opt.trace.c_str(), "a")) {
            fprintf(f, "# gram_mma_kernel ST=%d multi=%d guard=%d gen=%d oddrun=%d warps=%d rs=%d upc=%d passes=%d rc=%d nstage=%d gx=%d rows=%llu second=%d\n",
                    ST, (int)MULTI, (int)GUARD, (int)GEN, g.oddrun, g.warps, g.rs, g.upc, g.passes, g.rc, g.nstage, gx,
                    (unsigned long long)rows, g.second);
            fclose(f);
        }
    }
    // (without the second-order block only the block rows holding f(M_1), f(M_2) -- coordinates < 2l -- exist in the image)
    gram_mma_scatter_kernel<<<(unsigned)(((size_t)g.m * (g.m + 1) / 2 + 4 * g.l + 7) / 8), 256, 0, c->stream>>>(g.m, g.mpad, g.l, g.second ? g.m : 8 * g.imax, gx,
                                                                                 (const double *)c->block_buf.p, partials);
    c->launches++;
    VS_CUDA(cudaGetLastError());
    return VS_OK;
}

// Returns VS_OK with *handled = true when the tensor path ran; *handled = false means "use gram_kernel".
int launch_gram_mma(vs_ctx *c, int k, int l, uint64_t rows, const double *fvals, const double *shift_dev, int flags,
                    double *partials, bool *handled) {
    *handled = false;
    if ((reinterpret_cast<uintptr_t>(fvals) & 15) || rows == 0 || l < 1) return VS_OK;
    if (c->opt.gram_mma == 0) return VS_OK;
    MmaGeom g{};
    g.l = l;
    g.nt = 2 + 2 * k;
    g.m = g.nt * l;
    g.oddrun = (int)((rows & 1) && (l & 1));                 // rows * l odd: odd value blocks start 8 bytes off a 16-byte boundary
    g.gen = (l != 1 || (rows & 1)) ? 1 : 0;
    if (g.gen && c->opt.gram_mma_gen == 0) return VS_OK;     // VS_GRAM_GEN=0: register-tile kernel for l > 1 / odd rows
    g.nb = (g.m + 7) / 8;
    g.mpad = 8 * g.nb;
    g.second = (flags & VS_FLAG_SECOND_ORDER) ? 1 : 0;
    g.imax = g.second ? g.nb : (2 * l + 7) / 8;              // first order only: the rows of f(M_1), f(M_2) (coordinates < 2l)
    if (rows >= (1ull << 36) / (uint64_t)l) return VS_OK;
    // One diagonal super-tile of side ST >= nb when the whole matrix fits one warp's accumulators (k <= 23); otherwise
    // ST x ST super-tiles, ST in {4, 2} picked by a cost model fitted to B200 measurements (profiles/r01_gram_mma.txt):
    // a warp retires one DMMA per 60-80 cycles whatever else runs, so a pass costs (8x8 tiles of the heaviest super-tile /
    // warps sharing it) * that, or the bulk copies of the pass (~2 cycles per coordinate and 4-row step), whichever is larger.
    const bool multi = g.nb > 6;
    int ST = g.nb <= 2 ? 2 : g.nb == 3 ? 3 : g.nb == 4 ? 4 : 6;
    // consumer warps (+ 1 producer warp): 12 warps -> 168 registers per thread, 16 -> 128; the 2 x 2 form also runs with 32
    // warps (64 registers) -- used only where that turns two passes over the data into one (16..31 super-tiles: k = 50
    // 2.24 -> 2.05 ms); elsewhere the 15-warp form measured faster (k = 30: 0.76 vs 0.79 ms, k = 100: 1.95 vs 2.17,
    // l = 3 k = 20: 0.67 vs 0.87; tools/gram_probe.py).
    auto maxw_of = [&](int st) {
        if (!multi) return 11;
        const int nsb = (g.nb + st - 1) / st, nunits = g.second ? nsb * (nsb + 1) / 2 : nsb;
        const bool wide = st == 2 && nunits > 15 && nunits <= 31 && c->opt.gram_warps != 15;
        return (wide || c->opt.gram_warps == 31) && st == 2 ? 31 : 15;
    };
    if (multi) {
        double best = 0.0;
        for (int st : {4, 2}) {
            const int maxw = maxw_of(st);
            const int nsb = (g.nb + st - 1) / st;
            const int nunits = g.second ? nsb * (nsb + 1) / 2 : nsb;
            const int upc = nunits < maxw ? nunits : maxw, passes = (nunits + upc - 1) / upc, rs = maxw / upc;
            const int heavy = (g.second && nsb > 1) ? st * st : st * (st + 1) / 2;
            const double mma = (double)heavy / rs * (st == 4 ? 60.0 : 80.0), copy = 2.0 * g.m;
            const double cost = passes * (mma > copy ? mma : copy);
            if (nunits <= 128 && (best == 0.0 || cost < best)) { best = cost; ST = st; }
        }
        if (best == 0.0) return VS_OK;            // more super-tiles than the tables hold: register-tile kernel
    }
    if (multi && (c->opt.gram_st == 2 || c->opt.gram_st == 4)) ST = c->opt.gram_st;                  // tuning switch (VS_GRAM_ST)
    if (multi && 2 * l > 8 * ST) ST = 4;                      // the shifted sums (coordinates < 2l) live in super-tile (0, 0)
    if (2 * l > 8 * ST) return VS_OK;
    const int maxw = maxw_of(ST);
    const bool guard = multi || !g.second || g.nb != ST;
    g.nsb = (g.nb + ST - 1) / ST;
    g.nunits = g.second ? g.nsb * (g.nsb + 1) / 2 : g.nsb;
    g.upc = g.nunits < maxw ? g.nunits : maxw;
    g.passes = (g.nunits + g.upc - 1) / g.upc;
    g.rs = maxw / g.upc;
    g.warps = g.upc * g.rs;
    if (g.nunits > 128) return VS_OK;
    {
        // super-tiles, heaviest (most 8x8 tiles) first; then the items of a pass onto the sub-partitions, longest first
        struct Unit { int I, J, w; };
        std::vector<Unit> units;
        for (int I = 0; I < (g.second ? g.nsb : 1); ++I)
            for (int J = I; J < g.nsb; ++J) {
                int w = 0;
                for (int x = 0; x < ST; ++x)
                    for (int y = 0; y < ST; ++y) {
                        const int bi = ST * I + x, bj = ST * J + y;
                        if (bi < g.imax && bj < g.nb && bi <= bj) ++w;
                    }
                units.push_back({I, J, w});
            }
        std::stable_sort(units.begin(), units.end(), [](const Unit &a, const Unit &b) { return a.w > b.w; });
        for (int q = 0; q < g.nunits; ++q) {
            g.ui[q] = (unsigned char)units[q].I;
            g.uj[q] = (unsigned char)units[q].J;
            if (units[q].I == 0 && units[q].J == 0) g.sumu = q;
        }
        int load[4] = {0, 0, 0, 0}, used[4] = {0, 0, 0, 0};
        if (g.warps % 4 == 3) load[3] = 1;                           // the producer warp shares sub-partition (warps % 4)
        for (int w = 0; w < 32; ++w) g.witem[w] = 255;
        for (int item = 0; item < g.upc * g.rs; ++item) {
            const int wt = units[item / g.rs].w;                     // pass 0 decides; later passes have the same shape or lighter
            int best = -1;
            for (int sp = 0; sp < 4; ++sp) {
                const int slot = sp + 4 * used[sp];
                if (slot >= g.warps) continue;
                if (best < 0 || load[sp] < load[best]) best = sp;
            }
            g.witem[best + 4 * used[best]] = (unsigned char)item;
            used[best]++;
            load[best] += wt;
        }
    }
    const size_t avail = c->smem_optin;                       // 227 KB on sm_100a
    const size_t tail = ((size_t)g.upc * (8 * ST) * (8 * ST) + (size_t)g.rs * (g.gen ? ST : 1) * 64) * sizeof(double);
    // rows per chunk: as large as a ~60 KB stage allows (fewer, larger bulk copies and barrier round trips), ring of 3-6 stages
    int rc_cap = 256;
    if (c->opt.gram_rc > 0) rc_cap = c->opt.gram_rc;                                          // tuning switch (VS_GRAM_RC)
    size_t smem = 0;
    g.nstage = 0;
    for (int rc : {256, 128, 64, 32, 16, 8}) {
        if (rc > rc_cap && rc > 32) continue;
        if (rc < 32 && !g.gen) break;
        // doubles per staged row: rc (GEN: rc * l, + 2 for a misaligned start and the 16-byte round-up), pitch = 4 mod 16
        const int need = g.gen ? rc * l + 2 : rc;
        const int pitch = ((need + 11) / 16) * 16 + 4;
        const size_t stage = (size_t)(g.gen ? g.nt + 1 : g.mpad) * pitch * sizeof(double);
        int ns = (int)((avail - 2048) / stage);                 // one CTA per SM: the ring is what keeps HBM busy
        if (ns > 6) ns = 6;
        if ((stage > 60 * 1024 || ns < 3) && rc > (g.gen ? 8 : 32)) continue;
        if (ns < 2) break;
        g.rc = rc;
        g.pitch = pitch;
        g.nstage = ns;
        smem = MMA_BAR_DOUBLES * sizeof(double) + (size_t)ns * stage;
        break;
    }
    if (g.nstage < 2) return VS_OK;
    if (c->opt.gram_stages >= 1 && c->opt.gram_stages < g.nstage) g.nstage = c->opt.gram_stages;
    g.debug = c->opt.gram_debug;
    if (smem < MMA_BAR_DOUBLES * sizeof(double) + tail) smem = MMA_BAR_DOUBLES * sizeof(double) + tail;
    if (smem > avail) return VS_OK;
    int rc = VS_OK;
#define VS_MMA_CASE(S, M, G)                                                                       \
    rc = g.gen ? launch_mma_t<S, M, G, true>(c, g, smem, rows, fvals, shift_dev, partials)         \
               : launch_mma_t<S, M, G, false>(c, g, smem, rows, fvals, shift_dev, partials)
    if (multi) { if (ST == 4) VS_MMA_CASE(4, true, true); else VS_MMA_CASE(2, true, true); }
    else if (ST == 2) { if (guard) VS_MMA_CASE(2, false, true); else VS_MMA_CASE(2, false, false); }
    else if (ST == 3) { if (guard) VS_MMA_CASE(3, false, true); else VS_MMA_CASE(3, false, false); }
    else if (ST == 4) { if (guard) VS_MMA_CASE(4, false, true); else VS_MMA_CASE(4, false, false); }
    else { if (guard) VS_MMA_CASE(6, false, true); else VS_MMA_CASE(6, false, false); }
#undef VS_MMA_CASE
    if (rc == VS_OK) *handled = true;
    return rc;
}

}  // namespace vs
