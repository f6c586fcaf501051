// Objective evaluation to HBM (two-phase path), Gram/partial-sum reduction of given values, finalisation.
#include "device.cuh"

#include <cstdio>
#include <type_traits>
#include <vector>

namespace vs {

// ---------------------------------------------------------------------------------------------
// Two-phase path, phase 1: objective values of base rows, sample rows generated on the fly.
// One thread per (base row, point chunk).  The row's A_i / B_i live in shared memory, transposed
// ([coordinate][thread]) so every access is conflict-free; a point of the design is a *view*
// (base row, one substituted column) -- the 2+2k sample rows are never materialised.
// Replaces varsens/saltelli.py:308-353.  Used for heavy functors (RK4: one trajectory per thread)
// and for any k the fused kernel does not cover.
// ---------------------------------------------------------------------------------------------
struct SmemPoint {
    const double *base, *other;
    int j, stride;
    __device__ __forceinline__ double operator[](int c) const { return (c == j ? other : base)[c * stride]; }
};

template <class F, class = void> struct has_product_form : std::false_type {};
template <class F> struct has_product_form<F, std::enable_if_t<F::product_form>> : std::true_type {};

template <class F>
__global__ void eval_values_kernel(int k, int pts_per_chunk, SourceDev src, ScaleDev s, F f, uint64_t i_begin, uint64_t i_end,
                                   double *__restrict__ fvals) {
    extern __shared__ double smem[];
    const int nthr = blockDim.x;
    double *A = smem + threadIdx.x;                       // A[c*nthr]
    double *B = smem + (size_t)k * nthr + threadIdx.x;
    const uint64_t rows = i_end - i_begin;
    const uint64_t r = (uint64_t)blockIdx.x * nthr + threadIdx.x;
    if (r >= rows) return;
    const uint64_t i = i_begin + r;
    const uint64_t pi = src.perm[i];
    for (int c = 0; c < k; ++c) {
        A[c * nthr] = apply_scale(s, c, source_a(src, k, i, c));
        B[c * nthr] = apply_scale(s, c, source_b(src, k, pi, c));
    }
    const int npts = 2 + 2 * k;
    int p0 = blockIdx.y * pts_per_chunk, p1 = p0 + pts_per_chunk;
    if (p1 > npts) p1 = npts;
    if constexpr (has_product_form<F>::value) {
        // Product-form functors, f(x) = prod_c term(c, x_c) taken left to right from 1.0 (F::operator()).  The design
        // points of a row differ from M_1[i] / M_2[i] in one column, so their left-to-right products share the prefix
        // prod_{c<j}: the 2k terms are evaluated once per row (they replace the coordinates in shared memory) and point j
        // continues from the running prefix -- k(k-1)/2 multiplies per family instead of k^2 term evaluations, and bit for
        // bit the value F::operator() returns, because every product is still formed in ascending c.
        // (Six-points-at-a-time evaluation of every term: 25.4 ms for k = 50, n = 2^22; one point at a time: 29.5 ms.)
        for (int c = 0; c < k; ++c) {
            A[c * nthr] = f.term(c, A[c * nthr]);
            B[c * nthr] = f.term(c, B[c * nthr]);
        }
        auto store = [&](int P, double v) {
            if (P >= p0 && P < p1) fvals[(uint64_t)P * rows + r] = v;
        };
        double pa = 1.0, pb = 1.0;                       // prod_{c<j} term(c, A_c), prod_{c<j} term(c, B_c)
        for (int j = 0; j < k; ++j) {
            const double ta = A[j * nthr], tb = B[j * nthr];
            double vj = pb * ta;                         // N_j[j]  : M_2 with column j from M_1
            double vn = pa * tb;                         // N_nj[j] : M_1 with column j from M_2
            for (int c = j + 1; c < k; ++c) {
                vj *= B[c * nthr];
                vn *= A[c * nthr];
            }
            store(2 + j, vj);
            store(2 + k + j, vn);
            pa *= ta;
            pb *= tb;
        }
        store(0, pa);
        store(1, pb);
    } else {
        for (int p = p0; p < p1; ++p) {
            SmemPoint x;
            x.stride = nthr;
            if (p == 0) { x.base = A; x.other = A; x.j = -1; }
            else if (p == 1) { x.base = B; x.other = B; x.j = -1; }
            else if (p < 2 + k) { x.base = B; x.other = A; x.j = p - 2; }          // N_j[j]  : M_2 with col j from M_1
            else { x.base = A; x.other = B; x.j = p - 2 - k; }                      // N_nj[j] : M_1 with col j from M_2
            fvals[(uint64_t)p * rows + r] = f(x, k);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Two-phase path, phase 1, product-form functors (f(x) = prod_c term(c, x_c): the g-function), any k that fits.
// A CTA (8 warps) works on 32 base rows at a time, lane = row:
//   P1  warp w takes dimensions w, w+8, ...: Halton digit sums of A_i and B_i as two independent chains with warp-uniform base
//       (terms of the bases < 37 from a small shared table, terms of the larger bases COMPUTED from double-double reciprocals --
//       bit-identical to the table, host.cu: build_arith -- so no 160 KB table has to live in shared memory), scaling, and the
//       functor's term -> TA[d][row], TB[d][row];
//   P2  four warps run the four product chains over d (lane = row): prefix of TA, prefix of TB, suffix of TA, suffix of TB;
//   P3  warp w takes j = w, w+8, ...: f(N_j[j]) = PB[j] * TA[j] * SB[j+1], f(N_nj[j]) = PA[j] * TB[j] * SA[j+1], stored as
//       256-byte coalesced runs of the t-major value layout; f(M_1) = PA[k], f(M_2) = PB[k].
// O(k) multiplies per row instead of the O(k^2) of point-by-point evaluation: C4's second-order block went from 13 ms in
// this phase to ~1.5 (tools/bench_configs.py).  The values are the same products associated differently (prefix * term *
// suffix instead of left to right): <= 2 ulp from F::operator(), far inside the 1e-10 contract on the indices.
// ---------------------------------------------------------------------------------------------

// NR row groups per lane: a CTA tile has 32 NR rows and 8 NR warps.  NR = 2 (one CTA of 16 warps per SM instead of two of 8)
// keeps the rows in flight per SM, doubles the independent digit chains per warp and halves the per-dimension prologue per row
// in P1 -- and measured slower (see launch_eval_pf), so NR = 1 is the default and NR = 2 a switch.
template <class F, int NR>
__global__ void __launch_bounds__(256 * NR, NR == 1 ? 2 : 1)
eval_values_pf_kernel(int k, SourceDev src, ScaleDev s, F f, uint64_t i_begin, uint64_t i_end, uint32_t table_len, double *__restrict__ fvals) {
    constexpr int ROWS = 32 * NR, WARPS = 8 * NR;
    extern __shared__ __align__(16) double smem[];
    // layout: generator prefix (device.cuh: halton_prefix) | TA TB [k][ROWS] | PA PB SA SB [k+1][ROWS]
    const HaltonPrefix gen = halton_prefix(smem, k, src, s, table_len, !src.raw, src.raw ? 0 : WARPS);
    const HaltonShared &hs = gen.hs;
    double *TA = gen.table + table_len, *TB = TA + (size_t)k * ROWS;
    double *PA = TB + (size_t)k * ROWS, *PB = PA + (size_t)(k + 1) * ROWS, *SA = PB + (size_t)(k + 1) * ROWS, *SB = SA + (size_t)(k + 1) * ROWS;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint64_t rows = i_end - i_begin, n = src.n;
    const uint64_t ntiles = (rows + ROWS - 1) / ROWS;
    // base row of the lane's r-th row of a tile (clamped: the last tile may be ragged) and its permutation entry; the entry of
    // the NEXT tile is requested before P1 of the current one, so its DRAM latency (7 % of the stall samples when it was
    // loaded at the top of the loop, profiles/r02_evalpf_sass_profile_final.txt) is hidden behind a whole tile of work
    auto base_row = [&](uint64_t tile, int r) {
        const uint64_t q = tile * ROWS + 32 * r + lane;
        return i_begin + (q < rows ? q : rows - 1);
    };
    uint64_t pi_next[NR];
#pragma unroll
    for (int r = 0; r < NR; ++r) pi_next[r] = blockIdx.x < ntiles ? src.perm[base_row(blockIdx.x, r)] : 0;
    for (uint64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        // the lane's NR rows: tile * ROWS + 32 r + lane
        uint64_t rr[NR], ii[NR], pi[NR];
        bool live[NR];
        uint32_t ia[NR], ib[NR];
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            rr[r] = tile * ROWS + 32 * r + lane;
            live[r] = rr[r] < rows;
            ii[r] = base_row(tile, r);
            pi[r] = pi_next[r];
            ia[r] = (uint32_t)(src.start + ii[r]);
            ib[r] = (uint32_t)(src.start + n + pi[r]);
        }
        if (tile + gridDim.x < ntiles) {
#pragma unroll
            for (int r = 0; r < NR; ++r) pi_next[r] = src.perm[base_row(tile + gridDim.x, r)];
        }
        // ---- P1: coordinates and terms
        auto emit = [&](int d, int r, double pa, double pb) {
            if (s.kind == VS_SCALE_LINEAR) {
                pa = scale_value(VS_SCALE_LINEAR, gen.lb[d], gen.wr[d], pa);
                pb = scale_value(VS_SCALE_LINEAR, gen.lb[d], gen.wr[d], pb);
            } else if (s.kind == VS_SCALE_POWER) {
                pa = scale_value(VS_SCALE_POWER, gen.lb[d], gen.wr[d], pa);
                pb = scale_value(VS_SCALE_POWER, gen.lb[d], gen.wr[d], pb);
            }
            TA[(size_t)d * ROWS + 32 * r + lane] = f.term(d, pa);
            TB[(size_t)d * ROWS + 32 * r + lane] = f.term(d, pb);
        };
        if (src.raw) {
            for (int d = warp; d < k; d += WARPS)
#pragma unroll
                for (int r = 0; r < NR; ++r) emit(d, r, src.raw[ii[r] * (uint64_t)k + d], src.raw[(n + pi[r]) * (uint64_t)k + d]);
        } else {
            // units of one table dimension or two computed-term dimensions, balanced over the warps (device.cuh: halton_schedule)
            halton_units<NR>(warp, gen.ulist, k, ia, ib, hs, emit);
        }
        __syncthreads();
        // ---- P2: four product chains per row group, lane = row
        if (warp < 4 * NR) {
            const int rg = warp >> 2, ch = warp & 3, col = 32 * rg + lane;
            const double *Tm = (ch & 1) ? TB : TA;
            if (ch < 2) {
                double *P = ch ? PB : PA;
                double p = 1.0;
                P[col] = p;
                for (int c = 0; c < k; ++c) { p *= Tm[(size_t)c * ROWS + col]; P[(size_t)(c + 1) * ROWS + col] = p; }
            } else {
                double *S = (ch & 1) ? SB : SA;
                double p = 1.0;
                S[(size_t)k * ROWS + col] = p;
                for (int c = k - 1; c >= 0; --c) { p *= Tm[(size_t)c * ROWS + col]; S[(size_t)c * ROWS + col] = p; }
            }
        }
        __syncthreads();
        // ---- P3: the 2 + 2k values of every row
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            if (!live[r]) continue;
            const int col = 32 * r + lane;
            const uint64_t ro = rr[r];
            if (warp == 0) fvals[ro] = PA[(size_t)k * ROWS + col];                                  // f(M_1[i])
            if (warp == 1) fvals[rows + ro] = PB[(size_t)k * ROWS + col];                           // f(M_2[i])
            for (int j = warp; j < k; j += WARPS) {
                const double vj = PB[(size_t)j * ROWS + col] * TA[(size_t)j * ROWS + col] * SB[(size_t)(j + 1) * ROWS + col];   // M_2 with column j from M_1
                const double vn = PA[(size_t)j * ROWS + col] * TB[(size_t)j * ROWS + col] * SA[(size_t)(j + 1) * ROWS + col];   // M_1 with column j from M_2
                fvals[(uint64_t)(2 + j) * rows + ro] = vj;
                fvals[(uint64_t)(2 + k + j) * rows + ro] = vn;
            }
        }
        __syncthreads();
    }
}

template <class F, int NR>
static int launch_eval_pf_t(vs_ctx *c, int k, const SourceDev &src, const ScaleDev &s, const F &f, uint64_t i_begin, uint64_t i_end,
                            uint32_t table_len, size_t smem, double *fvals) {
    const uint64_t rows = i_end - i_begin;
    VS_CUDA(cudaFuncSetAttribute(eval_values_pf_kernel<F, NR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const uint64_t ntiles = (rows + 32 * NR - 1) / (32 * NR);
    const int per_sm = (NR == 1 && smem * 2 + 2048 <= c->smem_optin) ? 2 : 1;
    const unsigned grid = (unsigned)(ntiles < (uint64_t)(per_sm * c->sm_count) ? ntiles : (uint64_t)(per_sm * c->sm_count));
    time_begin(c);
    eval_values_pf_kernel<F, NR><<<grid, 256 * NR, smem, c->stream>>>(k, src, s, f, i_begin, i_end, table_len, fvals);
    time_end(c);
    c->launches++;
    VS_CUDA(cudaGetLastError());
    if (!c->opt.trace.empty()) {                      // VS_TRACE: the form that ran; tiles per CTA = ceil(ntiles / grid)
        if (FILE *fp = fopen(c->opt.trace.c_str(), "a")) {
            fprintf(fp, "# eval_values_pf_kernel NR=%d grid=%u ntiles=%llu rows=%llu\n", NR, grid, (unsigned long long)ntiles,
                    (unsigned long long)rows);
            fclose(fp);
        }
    }
    return VS_OK;
}

template <class F>
static int launch_eval_pf(vs_ctx *c, int k, const SourceDev &src, const ScaleDev &s, const F &f, uint64_t i_begin, uint64_t i_end,
                          double *fvals, bool *done) {
    *done = false;
    const uint64_t rows = i_end - i_begin;
    if (rows == 0 || c->opt.no_pf_eval) return VS_OK;
    if (!src.raw && (src.h.mode == VS_HALTON_HORNER || !src.h.arith_ok || halton_unit_count(k) > HL_MAX_UNITS)) return VS_OK;
    const uint32_t table_len = src.raw ? 0 : halton_table_prefix(c->halton);
    auto smem_of = [&](int nr) {
        return (halton_prefix_doubles(k) + table_len + 2 * (size_t)k * 32 * nr + 4 * (size_t)(k + 1) * 32 * nr + 2) * sizeof(double);
    };
    // VS_PF_ROWS=64: two row groups per lane (64-row tiles, one CTA of 16 warps per SM).  Measured SLOWER at C4 (3.07 vs 2.76 ms):
    // twice the independent chains per warp do not make up for losing the second CTA whose phases interleave with the first.
    const bool two = c->opt.pf_rows == 64 && smem_of(2) <= c->smem_optin && rows >= 64ull * c->sm_count;
    const size_t smem = smem_of(two ? 2 : 1);
    if (smem > c->smem_optin) return VS_OK;
    if (two) VS_TRY((launch_eval_pf_t<F, 2>(c, k, src, s, f, i_begin, i_end, table_len, smem, fvals)));
    else VS_TRY((launch_eval_pf_t<F, 1>(c, k, src, s, f, i_begin, i_end, table_len, smem, fvals)));
    *done = true;
    return VS_OK;
}

template <class F>
static int launch_eval_t(vs_ctx *c, int k, bool heavy, const SourceDev &src, const ScaleDev &s, const F &f, uint64_t i_begin,
                         uint64_t i_end, double *fvals) {
    uint64_t rows = i_end - i_begin;
    if (rows == 0) return VS_OK;
    int nthr = 128;
    while (nthr > 32 && 2 * (size_t)k * nthr * sizeof(double) > 96 * 1024) nthr >>= 1;
    size_t smem = 2 * (size_t)k * nthr * sizeof(double);
    VS_REQUIRE(smem <= c->smem_optin, VS_ERR_UNSUPPORTED, "k=%d does not fit shared memory", k);
    if (smem > 48 * 1024) VS_CUDA(cudaFuncSetAttribute(eval_values_kernel<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int npts = 2 + 2 * k;
    int ppc = heavy ? 1 : npts;
    dim3 grid((unsigned)((rows + nthr - 1) / nthr), (unsigned)((npts + ppc - 1) / ppc));
    time_begin(c);
    eval_values_kernel<F><<<grid, nthr, smem, c->stream>>>(k, ppc, src, s, f, i_begin, i_end, fvals);
    time_end(c);
    c->launches++;
    VS_CUDA(cudaGetLastError());
    if (!c->opt.trace.empty()) {                      // VS_TRACE: the form that ran (block size, points per thread, grid)
        if (FILE *fp = fopen(c->opt.trace.c_str(), "a")) {
            fprintf(fp, "# eval_values_kernel nthr=%d ppc=%d gx=%u gy=%u smem=%zu rows=%llu\n", nthr, ppc, grid.x, grid.y, smem,
                    (unsigned long long)rows);
            fclose(fp);
        }
    }
    return VS_OK;
}

template <int S>
static int launch_rk4(vs_ctx *c, int k, const SourceDev &src, const ScaleDev &s, double dt, int nsteps, uint64_t i_begin,
                      uint64_t i_end, double *fvals) {
    RK4Chain<S> f{dt, nsteps};
    return launch_eval_t(c, k, true, src, s, f, i_begin, i_end, fvals);
}

int launch_eval_values(vs_ctx *c, int k, const SourceDev &src, const ScaleDev &s, const ObjectiveDev &o, uint64_t i_begin,
                       uint64_t i_end, double *fvals, bool count) {
    switch (o.id) {
    case VS_OBJ_GFUNCTION: {
        GFunction f{o.params + k, o.params + 2 * k};
        bool done = false;
        VS_TRY(launch_eval_pf(c, k, src, s, f, i_begin, i_end, fvals, &done));
        if (done) return VS_OK;
        return launch_eval_t(c, k, false, src, s, f, i_begin, i_end, fvals);
    }
    case VS_OBJ_ISHIGAMI: {
        const double *h = o.host;
        Ishigami f{h[0], h[1]};
        return launch_eval_t(c, k, false, src, s, f, i_begin, i_end, fvals);
    }
    case VS_OBJ_RK4_CHAIN: {
        const double *h = o.host;
        double dt = h[0];
        int ns = (int)h[1];
        switch (k / 2) {
#define VS_RK4_CASE(S) case S: return launch_rk4<S>(c, k, src, s, dt, ns, i_begin, i_end, fvals);
            VS_RK4_CASE(1) VS_RK4_CASE(2) VS_RK4_CASE(3) VS_RK4_CASE(4) VS_RK4_CASE(5) VS_RK4_CASE(6)
            VS_RK4_CASE(7) VS_RK4_CASE(8) VS_RK4_CASE(9) VS_RK4_CASE(10) VS_RK4_CASE(12) VS_RK4_CASE(16)
#undef VS_RK4_CASE
        default: {
            RK4ChainDyn f{dt, ns};
            return launch_eval_t(c, k, true, src, s, f, i_begin, i_end, fvals);
        }
        }
    }
    case VS_OBJ_MASS_ACTION:
    case VS_OBJ_MASS_ACTION_ADAPTIVE:
    case VS_OBJ_MASS_ACTION_STIFF:
        return launch_network_values(c, k, src, s, o, i_begin, i_end, fvals, count);
    }
    set_error("unknown objective id %d", o.id);
    return VS_ERR_ARG;
}

// ---------------------------------------------------------------------------------------------
// Estimator reductions on given values: symmetric Gram G = sum_i v_i v_i^T of the per-row vector
// v_i (m = (2+2k) l entries) + shifted sums for var_y.  Everything the estimators of
// varsens/saltelli.py:577-622 need is an entry of G (SURVEY.md §3.4: only 3 distinct k x k Grams).
//
// CTA: stages R rows of v in shared memory (coalesced loads of the t-major value layout), then
// every thread accumulates one T x T register tile of the upper triangle over a subset of the
// staged rows (2T shared loads per T^2 DFMA).  Row groups and CTAs are combined in a fixed order
// -> bit-reproducible results.
// ---------------------------------------------------------------------------------------------
template <int T>
__global__ void __launch_bounds__(256) gram_kernel(GramGeom g, uint64_t rows, const double *__restrict__ fvals,
                                                   const double *__restrict__ shift, double *__restrict__ blockpart) {
    extern __shared__ double smem[];
    double *Y = smem;  // [R][mp]
    const int tid = threadIdx.x;
    const int grp = tid / g.LG, tl = tid - grp * g.LG;
    const int tile = blockIdx.y * g.LG + tl;
    const bool active = (grp < g.RG) && (tile < g.ntiles);
    int tr = 0, tc = 0;
    if (active) tile_coords(tile, g.nt, tr, tc);
    double acc[T][T];
#pragma unroll
    for (int x = 0; x < T; ++x)
#pragma unroll
        for (int y = 0; y < T; ++y) acc[x][y] = 0.0;
    // shifted sums: thread e < 2l of pass 0 owns (t = e / l in {0,1}, o = e % l)
    const bool sum_thread = (blockIdx.y == 0) && (tid < 2 * g.l);
    const double my_shift = (sum_thread && shift) ? shift[tid % g.l] : 0.0;
    double sS = 0.0, sQ = 0.0;

    const uint64_t nchunks = (rows + g.R - 1) / g.R;
    for (uint64_t ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
        const uint64_t r0 = ch * g.R;
        const int valid = (int)((rows - r0 < (uint64_t)g.R) ? rows - r0 : g.R);
        // stage: global element (t, r, o) at fvals[(t*rows + r0 + r)*l + o] -> Y[r][t*l + o]
        const int per_t = g.R * g.l;
        const int nT = g.m / g.l;
        // Loads first (4 independent requests in flight per thread), then the transposed stores: with one load per loop
        // trip the kernel sat on HBM latency (2.0 ms for 1.4 GB; this form: see profiles/r01_other_configs.json).
        const int total = nT * per_t;
        for (int e0 = tid; e0 < total; e0 += 4 * (int)blockDim.x) {
            double v[4];
            int dst[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int e = e0 + u * (int)blockDim.x;
                dst[u] = -1;
                v[u] = 0.0;
                if (e < total) {
                    int t = e / per_t, rem = e - t * per_t;
                    int r = rem / g.l, o = rem - r * g.l;
                    dst[u] = r * g.mp + t * g.l + o;
                    if (r < valid) v[u] = __ldg(fvals + ((uint64_t)t * rows + r0 + r) * g.l + o);
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (dst[u] >= 0) Y[dst[u]] = v[u];
        }
        for (int e = tid; e < g.R * (g.mp - g.m); e += blockDim.x) {   // zero the column padding
            int r = e / (g.mp - g.m), cidx = g.m + e % (g.mp - g.m);
            Y[r * g.mp + cidx] = 0.0;
        }
        __syncthreads();
        if (active) {
            for (int r = grp; r < g.R; r += g.RG) {
                const double *row = Y + r * g.mp;
                double a[T], b[T];
#pragma unroll
                for (int x = 0; x < T; ++x) { a[x] = row[tr * T + x]; b[x] = row[tc * T + x]; }
#pragma unroll
                for (int x = 0; x < T; ++x)
#pragma unroll
                    for (int y = 0; y < T; ++y) acc[x][y] = fma(a[x], b[y], acc[x][y]);
            }
        }
        if (sum_thread) {
            for (int r = 0; r < valid; ++r) {
                double d = Y[r * g.mp + tid] - my_shift;
                sS += d;
                sQ = fma(d, d, sQ);
            }
        }
        __syncthreads();
    }
    // combine row groups in fixed order through shared memory: red[grp][tl][T*T]
    double *red = smem;
    if (grp < g.RG && tl < g.LG) {
#pragma unroll
        for (int x = 0; x < T; ++x)
#pragma unroll
            for (int y = 0; y < T; ++y) red[((size_t)grp * g.LG + tl) * (T * T) + x * T + y] = acc[x][y];
    }
    __syncthreads();
    const size_t per_block = (size_t)g.passes * g.LG * (T * T) + 4 * (size_t)g.l;
    double *bp = blockpart + (size_t)blockIdx.x * per_block;
    for (int e = tid; e < g.LG * T * T; e += blockDim.x) {
        double s = 0.0;
        for (int q = 0; q < g.RG; ++q) s += red[(size_t)q * g.LG * (T * T) + e];
        bp[(size_t)blockIdx.y * g.LG * (T * T) + e] = s;
    }
    if (sum_thread) {
        double *ss = bp + (size_t)g.passes * g.LG * (T * T);
        ss[tid] = sS;                 // S_A[l], S_B[l]
        ss[2 * g.l + tid] = sQ;       // Q_A[l], Q_B[l]
    }
}

// Sum CTA partials in CTA order and scatter tile entries into the packed upper triangle.
__global__ void __launch_bounds__(256) gram_scatter_kernel(GramGeom g, int nblocks, const double *__restrict__ blockpart,
                                                           double *__restrict__ partials) {
    const int T = g.T;
    const size_t tile_elems = (size_t)g.passes * g.LG * (T * T);
    const size_t per_block = tile_elems + 4 * (size_t)g.l;
    const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t nthreads = (size_t)gridDim.x * blockDim.x;
    for (size_t e = gid; e < per_block; e += nthreads) {
        double s = 0.0;
        int b = 0;
        for (; b + 8 <= nblocks; b += 8) {               // 8 loads in flight, added in CTA order (bit-reproducible)
            double v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = blockpart[(size_t)(b + u) * per_block + e];
#pragma unroll
            for (int u = 0; u < 8; ++u) s += v[u];
        }
        for (; b < nblocks; ++b) s += blockpart[(size_t)b * per_block + e];
        if (e >= tile_elems) {
            partials[e - tile_elems] = s;
            continue;
        }
        int slot = (int)(e / (T * T)), within = (int)(e % (T * T));
        int pass = slot / g.LG, tl = slot % g.LG;
        int tile = pass * g.LG + tl;
        if (tile >= g.ntiles) continue;
        int tr, tc;
        tile_coords(tile, g.nt, tr, tc);
        int p = tr * T + within / T, q = tc * T + within % T;
        if (p >= g.m || q >= g.m || p > q) continue;
        size_t off = 4 * (size_t)g.l + (size_t)p * g.m - (size_t)p * (p - 1) / 2 + (size_t)(q - p);
        partials[off] = s;
    }
}

int launch_gram_scatter(vs_ctx *c, const GramGeom &g, int nblocks, const double *blockpart, double *partials, int plen);

static GramGeom make_geom(int k, int l, int flags, int T) {
    GramGeom g{};
    g.l = l;
    g.m = (2 + 2 * k) * l;
    g.T = T;
    g.nt = (g.m + T - 1) / T;
    g.mp = g.nt * T;
    if (g.mp % 2 == 0) g.mp += 1;
    g.tr_max = (flags & VS_FLAG_SECOND_ORDER) ? g.nt : (2 * l + T - 1) / T;
    if (g.tr_max > g.nt) g.tr_max = g.nt;
    g.ntiles = 0;
    for (int tr = 0; tr < g.tr_max; ++tr) g.ntiles += g.nt - tr;
    int lg = ((g.ntiles + 31) / 32) * 32;
    if (lg > 256) lg = 256;
    g.LG = lg;
    g.RG = 256 / lg;
    g.passes = (g.ntiles + lg - 1) / lg;
    int R = (int)((64 * 1024) / ((size_t)g.mp * sizeof(double)));
    if (R > 64) R = 64;
    if (R < g.RG) R = g.RG;
    R = (R / g.RG) * g.RG;
    g.R = R;
    return g;
}

static double geom_cost(const GramGeom &g) {
    // DFMA issue slots per staged row, per CTA (lower is better)
    return (double)g.passes * g.LG * g.T * g.T / (double)(g.RG);
}

template <int T>
static int launch_gram_t(vs_ctx *c, const GramGeom &g, uint64_t rows, const double *fvals, const double *shift_dev,
                         double *partials, int plen) {
    size_t smem_stage = (size_t)g.R * g.mp * sizeof(double);
    size_t smem_red = (size_t)g.RG * g.LG * T * T * sizeof(double);
    size_t smem = smem_stage > smem_red ? smem_stage : smem_red;
    VS_REQUIRE(smem <= c->smem_optin, VS_ERR_UNSUPPORTED, "Gram tile needs %zu bytes of shared memory", smem);
    VS_CUDA(cudaFuncSetAttribute(gram_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    uint64_t nchunks = (rows + g.R - 1) / g.R;
    // as many CTAs per SM as shared memory allows (up to 8): the staging loads need memory-level parallelism
    int per_sm = (int)((c->smem_optin > 0 ? (size_t)200 * 1024 : (size_t)48 * 1024) / (smem + 1024));
    if (per_sm > 8) per_sm = 8;
    if (per_sm < 1) per_sm = 1;
    int gx = (int)(nchunks < (uint64_t)(per_sm * c->sm_count) ? nchunks : (uint64_t)(per_sm * c->sm_count));
    if (gx < 1) gx = 1;
    size_t per_block = (size_t)g.passes * g.LG * (T * T) + 4 * (size_t)g.l;
    VS_TRY(ensure(c, c->block_buf, (size_t)gx * per_block * sizeof(double)));
    time_begin(c);
    gram_kernel<T><<<dim3(gx, g.passes), 256, smem, c->stream>>>(g, rows, fvals, shift_dev, (double *)c->block_buf.p);
    time_end(c);
    c->launches++;
    VS_CUDA(cudaGetLastError());
    if (!c->opt.trace.empty()) {                      // VS_TRACE: the form that ran; chunks per CTA = ceil(ceil(rows / R) / gx)
        if (FILE *f = fopen(c->opt.trace.c_str(), "a")) {
            fprintf(f, "# gram_kernel T=%d LG=%d RG=%d passes=%d R=%d gx=%d rows=%llu\n", T, g.LG, g.RG, g.passes, g.R, gx,
                    (unsigned long long)rows);
            fclose(f);
        }
    }
    return launch_gram_scatter(c, g, gx, (const double *)c->block_buf.p, partials, plen);
}

int launch_gram_scatter(vs_ctx *c, const GramGeom &g, int nblocks, const double *blockpart, double *partials, int plen) {
    VS_CUDA(cudaMemsetAsync(partials, 0, (size_t)plen * sizeof(double), c->stream));
    size_t per_block = (size_t)g.passes * g.LG * (g.T * g.T) + 4 * (size_t)g.l;
    int rb = (int)((per_block + 255) / 256);
    gram_scatter_kernel<<<rb, 256, 0, c->stream>>>(g, nblocks, blockpart, partials);
    c->launches++;
    VS_CUDA(cudaGetLastError());
    return VS_OK;
}

int launch_partials_from_values(vs_ctx *c, int k, int l, uint64_t rows, const double *fvals, const double *shift_dev,
                                int flags, double *partials) {
    int plen = (int)vs_partials_len(k, l);
    bool handled = false;
    VS_TRY(launch_gram_mma(c, k, l, rows, fvals, shift_dev, flags, partials, &handled));
    if (handled) return VS_OK;
    GramGeom best = make_geom(k, l, flags, 4);
    for (int T : {6, 8}) {
        GramGeom g = make_geom(k, l, flags, T);
        if (geom_cost(g) < geom_cost(best)) best = g;
    }
    switch (best.T) {
    case 4: return launch_gram_t<4>(c, best, rows, fvals, shift_dev, partials, plen);
    case 6: return launch_gram_t<6>(c, best, rows, fvals, shift_dev, partials, plen);
    default: return launch_gram_t<8>(c, best, rows, fvals, shift_dev, partials, plen);
    }
}

// ---------------------------------------------------------------------------------------------
// Finalisation: the estimators of varsens/saltelli.py:577-622 on the sufficient statistics, same
// operation order (E_2 over n; U and Grams over n-1; mixed normalisation is the reference's).
// Result buffer: see result_len (vs_internal.cuh).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) finalize_kernel(int k, int l, double n, double rows, const double *__restrict__ P, int second_order,
                                                       double *__restrict__ res) {
    finalize_body(k, l, n, rows, P, second_order, res);
}

// Partial-sum all-reduce over NVLink peer memory fused with the finalisation (see vs_allreduce_finalize_p2p); the stand-alone
// form of the exchange the fused kernel runs in its tail (fused_impl.cuh: fused_tail), for partial sums that come from elsewhere
// (two-phase path, user values).  Single CTA; same low-latency protocol (device.cuh: ll_push / ll_reduce).
// Status slot res[rlen + HOST_RES_STATUS] = 1.0 if a peer did not show up within timeout_ns (the indices are then meaningless),
// else 0.0.
__global__ void __launch_bounds__(256) p2p_reduce_finalize_kernel(int k, int l, double n, double rows, int world, int rank,
                                                                  const uint64_t *__restrict__ bufs, unsigned epoch, int plen, int rlen,
                                                                  unsigned long long timeout_ns, const double *__restrict__ mine,
                                                                  int second_order, double *__restrict__ reduced, double *__restrict__ res) {
    __shared__ unsigned timed_out;
    if (threadIdx.x == 0) timed_out = 0u;
    __syncthreads();
    ll_push(bufs, world, rank, epoch, plen, mine);
    if (!ll_reduce(bufs, world, rank, epoch, plen, reduced, timeout_ns)) timed_out = 1u;
    __syncthreads();
    finalize_body(k, l, n, rows, reduced, second_order, res);
    if (threadIdx.x == 0) res[rlen + HOST_RES_STATUS] = timed_out ? 1.0 : 0.0;
}

int launch_p2p_reduce_finalize(vs_ctx *c, int k, int l, uint64_t n, uint64_t rows, int world, int rank, const uint64_t *peer_bufs_dev,
                               const uint64_t *peer_flags_dev, uint32_t epoch, const double *partials, int flags, double *res_dev) {
    const int plen = (int)vs_partials_len(k, l);
    VS_TRY(ensure(c, c->part_buf, (size_t)plen * sizeof(double)));
    VS_REQUIRE(partials < (const double *)c->part_buf.p || partials >= (const double *)c->part_buf.p + plen, VS_ERR_ARG,
               "partials_dev must not alias the exchange scratch");
    (void)peer_flags_dev;
    p2p_reduce_finalize_kernel<<<1, 256, 0, c->stream>>>(k, l, (double)n, (double)rows, world, rank, peer_bufs_dev, epoch,
                                                          plen, (int)result_len(k, l), (unsigned long long)c->opt.p2p_timeout_ms * 1000000ull,
                                                          partials, (flags & VS_FLAG_SECOND_ORDER) ? 1 : 0,
                                                          (double *)c->part_buf.p, res_dev);
    c->launches++;
    VS_CUDA(cudaGetLastError());
    return VS_OK;
}

int launch_finalize(vs_ctx *c, int k, int l, uint64_t n, uint64_t rows, const double *partials, int flags, double *res_dev) {
    finalize_kernel<<<1, 256, 0, c->stream>>>(k, l, (double)n, (double)rows, partials, (flags & VS_FLAG_SECOND_ORDER) ? 1 : 0, res_dev);
    c->launches++;
    VS_CUDA(cudaGetLastError());
    return VS_OK;
}

}  // namespace vs
