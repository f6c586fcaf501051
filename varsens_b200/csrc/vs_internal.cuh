// Internal declarations shared by the translation units of libvarsens_b200.so.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/varsens_b200.h"

namespace vs {

// ---------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------
void set_error(const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what, const char *file, int line);

#define VS_CUDA(call)                                                              \
    do {                                                                           \
        cudaError_t e__ = (call);                                                  \
        if (e__ != cudaSuccess) return ::vs::cuda_fail(e__, #call, __FILE__, __LINE__); \
    } while (0)

#define VS_TRY(call)                \
    do {                            \
        int s__ = (call);           \
        if (s__ != VS_OK) return s__; \
    } while (0)

#define VS_REQUIRE(cond, code, ...)   \
    do {                              \
        if (!(cond)) {                \
            ::vs::set_error(__VA_ARGS__); \
            return (code);            \
        }                             \
    } while (0)

// ---------------------------------------------------------------------------------------------
// device-side descriptors (plain structs passed by value to kernels)
// ---------------------------------------------------------------------------------------------
// Halton term table: terms[off[d] + j*base[d] + digit] = digit / base[d]^(j+1) (host-built, fp64
// division; see vs_halton_terms).  magic[d] = floor(2^64 / base[d]) + 1 gives an exact quotient
// of any 32-bit index by one 64-bit mul-high.
struct HaltonDev {
    const double *terms;
    const uint32_t *base;
    const uint64_t *magic;
    const uint32_t *off;
    uint32_t total_terms;
    int mode;               // enum vs_halton_mode (HORNER: the table is not used)
    const double *fixed;    // the same terms in the fused kernels' fixed layout (all digit positions of a 32-bit index), k <= 32
    uint32_t fixed_len;
    const double *arh, *arl; // [k][HL_J] double-double reciprocals / 8 of the computed-term form (host.cu: build_arith), device
    int arith_ok;           // they reproduce the term table bit for bit
};
constexpr int HL_D0 = 11;   // run-time-base generators: dimensions >= HL_D0 (bases >= 37) compute their terms, below: table rows
constexpr int HL_J = 7;     // digit positions of a 32-bit index in base >= 37 (layout of HaltonDev::arh / arl)

// scale.py:33 / :62 lowered: linear  -> p * w + lb   (w = ub - lb rounded on the host, as numpy does)
//                            power   -> lb * pow(r, p) (r = ub / lb rounded on the host)
struct ScaleDev {
    int kind;
    const double *lb;
    const double *wr;
    const double *host;     // host copy: lb[k] | wr[k] (lives in the ctx)
};

// Where the unscaled points of the base design come from.
struct SourceDev {
    HaltonDev h;            // Halton (raw == nullptr)
    const double *raw;      // or an unscaled (2n,k) matrix
    const uint32_t *perm;   // row permutation of M_2
    uint64_t n;
    uint64_t start;         // Halton index of base row 0 of M_1: 20k + discard + 1
};

// Geometry of a tiled upper-triangular Gram accumulation (kernels_vals.cu, kernels_fused.cu).
// Tile `id` (row-major over tr < tr_max, tc >= tr) covers G[tr*T .. tr*T+T)[tc*T .. tc*T+T).
struct GramGeom {
    int m, l, T, nt, mp;        // mp = padded length of a staged row (odd -> conflict-free transposed stores)
    int ntiles, tr_max;
    int LG, RG;                 // lanes per tile group (multiple of 32), row groups per CTA
    int R;                      // rows staged per iteration
    int passes;
};

struct ObjectiveDev {
    int id;
    const double *params;   // device copy of the host params (plus derived values, see device.cuh)
    int n_params;
    const double *host;     // the same values on the host (lives in the ctx)
    int l = 1;              // outputs per point (L of a mass-action network)
};

// ---------------------------------------------------------------------------------------------
// host context
// ---------------------------------------------------------------------------------------------
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
};

struct HaltonCache {
    int k = 0;
    int mode = 0;
    std::vector<uint32_t> ndigits;
    std::vector<uint32_t> off;      // host copy of HaltonDev::off: dimension after dimension, base * ndigits terms each
    // double-double reciprocals for computed terms (fused_impl.cuh: digit_step_arith), [k][HL_J], and whether they reproduce
    // every entry of the term table bit for bit (checked when the table is built)
    std::vector<double> arh, arl;
    bool arith_ok = false;
    HaltonDev dev{};
    void *blob = nullptr;
};
// Doubles of the term table that hold the dimensions below HL_D0: what the run-time-base generators copy to shared memory.
inline uint32_t halton_table_prefix(const HaltonCache &hc) { return hc.k > HL_D0 ? hc.off[HL_D0] : hc.dev.total_terms; }

// Switches read from the environment ONCE, at vs_ctx_create (and again on vs_ctx_reload_env) -- never on a launch path.
struct Options {
    int fused_variant = 0;      // VS_FUSED_VARIANT  (0 = default choice per k)
    int no_pipeline = 0;        // VS_NO_PIPELINE    host permutation: one copy, then the launch (no chunk flags)
    std::string trace;          // VS_TRACE          file for CTA 0's clock stamps
    int gram_mma = -1;          // VS_GRAM_MMA       (-1 = default)
    int export_slow_gen = 0;    // VS_EXPORT_SLOW_GEN=1: generic digit loop in the bulk export kernel (comparison runs)
    int export_copies = 0;      // VS_EXPORT_COPIES=1|2: store warps / tile copies of the bulk export kernel (0: by window shape)
    int gram_mma_gen = -1;      // VS_GRAM_GEN       0: register-tile kernel for l > 1 outputs / odd row counts
    int pf_rows = 0;            // VS_PF_ROWS=64: 64-row tiles (two row groups per lane) in the product-form evaluation kernel (measured slower)
    int gram_warps = 0;         // VS_GRAM_WARPS=15|31: consumer warps of the 2 x 2 super-tile form (0: 31 where that saves a pass)
    int gram_st = 0, gram_rc = 0, gram_stages = 0, gram_debug = 0;
    int p2p_timeout_ms = 10000; // VS_P2P_TIMEOUT_MS bounded wait for the peers' flags in the exchange
    int halton_mode = 0;        // VS_HALTON_MODE    term-table arithmetic (enum vs_halton_mode)
    int index_bits = 0;         // VS_INDEX_BITS=32 forces the general (32-bit index) fused kernel
    int no_bulk_export = 0;     // VS_NO_BULK_EXPORT=1: export mode through the scalar-store kernel
    int no_pf_eval = 0;         // VS_NO_PF_EVAL=1: two-phase path evaluates product-form functors point by point (old kernel)
};

// What the tail of the fused kernel has to do after the CTA partial sums are complete (host side of FusedTail).
struct FusedReq {
    int mode = 0;                       // 0 = partial sums only, 1 = + estimators, 2 = + peer-memory all-reduce + estimators
    uint64_t n_total = 0, rows_total = 0;
    int world = 1, rank = 0;
    uint32_t epoch = 0;
    const uint64_t *peer_bufs_dev = nullptr, *peer_flags_dev = nullptr;
    int poll_perm = 0;                  // the permutation is copied into its staging buffer while the kernel runs (sentinel polling)
};

}  // namespace vs

struct vs_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;       // stream the kernels run on
    cudaStream_t own_stream = nullptr;
    cudaStream_t copy_stream = nullptr;  // H2D staging overlapped with compute
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool timing = false;                 // record events around the main kernel of each call (vs_ctx_set_timing)
    bool timed = false;
    uint64_t launches = 0;
    int sm_count = 0;
    size_t smem_optin = 0;
    vs::HaltonCache halton;
    // last uploaded descriptors: identical descriptors are not uploaded (or synchronised on) again
    std::vector<double> scale_host, obj_host;
    std::vector<uint64_t> peer_tab;
    vs::DevBuf peer_buf;
    vs::Options opt;
    double *host_res = nullptr;          // mapped pinned host memory the fused kernel's tail writes the results to
    size_t host_res_cap = 0;             // doubles
    vs::DevBuf ticket_buf;               // ticket counters of the fused kernel's two-level combine (64 x uint32, zero between launches)
    vs::DevBuf poll_buf;                 // staging buffer of a host permutation that is polled while it arrives: all entries hold the
    bool poll_clean = false;             // sentinel 0xFFFFFFFF between calls (the kernel puts it back); false -> refill before use
    int scale_kind_cached = -1, scale_k_cached = -1, obj_id_cached = -1;
    // scratch
    std::vector<cudaEvent_t> pipe_ev;    // [0]: "compute stream is done with the staging buffer" (ordering of the next H2D copy)
    vs::DevBuf pipe_buf;
    vs::DevBuf stats_buf;                // 4 x uint64 step counts of the last adaptive or stiff network evaluation (vs_last_network_stats)
    vs::DevBuf scale_buf, obj_buf, perm_buf, raw_buf, io_buf, part_buf, block_buf, res_buf, dir_buf, misc_buf;
};

namespace vs {

int ensure(vs_ctx *c, DevBuf &b, size_t bytes);
int get_halton(vs_ctx *c, int k, uint64_t max_index, HaltonDev *out);
int get_scale(vs_ctx *c, int k, const vs_scale *s, ScaleDev *out);
int get_objective(vs_ctx *c, int k, int objective, const double *params, int n_params, ObjectiveDev *out);
// Validation of (k, objective, params) without a ctx: the outputs per point in *l and, if h != nullptr, the parameter block
// get_objective uploads (host.cu).
int objective_host(int k, int objective, const double *params, int n_params, std::vector<double> *h, int *l);
// Returns a device pointer for an input buffer (staging a host buffer through `scratch`).
int stage_in(vs_ctx *c, DevBuf &scratch, const void *p, int mem, size_t bytes, const void **dev);
int make_source(vs_ctx *c, int k, uint64_t n, uint64_t discard, const uint32_t *perm, int perm_mem,
                uint64_t perm_begin, uint64_t perm_count, const double *raw, int raw_mem, SourceDev *out);
bool capturing(vs_ctx *c);
void time_begin(vs_ctx *c);
void time_end(vs_ctx *c);

// kernels_gen.cu
int launch_halton(vs_ctx *c, int k, uint64_t first, uint64_t count, const HaltonDev &h, const ScaleDev &s, double *out);
int launch_sobol(vs_ctx *c, int k, uint64_t first, uint64_t count, const uint32_t *dir_dev, int quantize6,
                 const ScaleDev &s, double *out);
int launch_sample_flat(vs_ctx *c, int k, const SourceDev &src, const ScaleDev &s, uint64_t row_begin,
                       uint64_t row_end, double *out);
int launch_sample_shard(vs_ctx *c, int k, const SourceDev &src, const ScaleDev &s, uint64_t i_begin, uint64_t i_end, double *out);
// kernels_vals.cu
// count = false: an adaptive or stiff network's step counts (vs_last_network_stats) are neither reset nor added to
int launch_eval_values(vs_ctx *c, int k, const SourceDev &src, const ScaleDev &s, const ObjectiveDev &o,
                       uint64_t i_begin, uint64_t i_end, double *fvals, bool count = true);
int launch_partials_from_values(vs_ctx *c, int k, int l, uint64_t rows, const double *fvals, const double *shift_dev,
                                int flags, double *partials);
int launch_finalize(vs_ctx *c, int k, int l, uint64_t n, uint64_t rows, const double *partials, int flags, double *res_dev);
int launch_p2p_reduce_finalize(vs_ctx *c, int k, int l, uint64_t n, uint64_t rows, int world, int rank, const uint64_t *peer_bufs_dev,
                               const uint64_t *peer_flags_dev, uint32_t epoch, const double *partials, int flags, double *res_dev);
int launch_gram_scatter(vs_ctx *c, const GramGeom &g, int nblocks, const double *blockpart, double *partials, int plen);
// kernels_gram_mma.cu: tensor-path Gram (*handled = false -> caller falls back to gram_kernel)
int launch_gram_mma(vs_ctx *c, int k, int l, uint64_t rows, const double *fvals, const double *shift_dev, int flags,
                    double *partials, bool *handled);
// kernels_network.cu: VS_OBJ_MASS_ACTION, VS_OBJ_MASS_ACTION_ADAPTIVE and VS_OBJ_MASS_ACTION_STIFF
int network_describe(int k, int objective, const double *params, int n_params, std::vector<double> *h, int *l);
int network_check_fit(vs_ctx *c, int k, const ObjectiveDev &o);       // VS_ERR_UNSUPPORTED if the state does not fit
int launch_network_values(vs_ctx *c, int k, const SourceDev &src, const ScaleDev &s, const ObjectiveDev &o, uint64_t i_begin,
                          uint64_t i_end, double *fvals, bool count);
// kernels_fused.cu
bool fused_supported(int k, int objective, int flags);
// true if the kernel chosen for (k, objective, flags) runs the whole step in ONE launch (FusedReq modes 1/2, chunk flags)
bool fused_tail_supported(vs_ctx *c, int k, int objective, int flags);
// partials may be nullptr when req->mode >= 1.  *finalized reports whether the tail ran (results in c->host_res).
int launch_fused(vs_ctx *c, int k, const SourceDev &src, const ScaleDev &s, const ObjectiveDev &o, uint64_t i_begin,
                 uint64_t i_end, int flags, double *partials, const FusedReq *req, bool *finalized);
int ensure_host_res(vs_ctx *c, size_t doubles);
void load_options(Options &o);

// Result block, in this order: E_2[l] var_y[l] U_j[kl] U_nj[kl] sens[kl] sens_t[kl] sens_2[(kl)^2] sens_2n[(kl)^2], always
// sized for the second-order form.  In the ctx's mapped host buffer HOST_RES_EXTRA doubles follow it: the status slot
// (written by the fused kernel's tail and the stand-alone exchange kernel) and the time stamps of the fused kernel's tail.
__host__ __device__ constexpr size_t result_len(int k, int l) {
    return 2 * (size_t)l + 4 * (size_t)k * l + 2 * ((size_t)k * l) * ((size_t)k * l);
}
constexpr int HOST_RES_EXTRA = 32;      // doubles after the results
constexpr int HOST_RES_STATUS = 0;      // offset after the results: 0.0 ok, 1.0 a peer did not publish within the time-out
constexpr int HOST_RES_STAMPS = 1;      // offset after the results of the 11 tail time stamps (ns, vs_last_tail_ns)
// microbench.cu
int launch_fp64_peak(vs_ctx *c, double *tflops);

}  // namespace vs
