// Context, error reporting, scratch management and host-built tables.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "vs_internal.cuh"

namespace vs {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char *what, const char *file, int line) {
    set_error("CUDA error %d (%s) at %s:%d in %s", (int)e, cudaGetErrorString(e), file, line, what);
    return VS_ERR_CUDA;
}

int ensure(vs_ctx *c, DevBuf &b, size_t bytes) {
    if (bytes <= b.cap && b.p) return VS_OK;
    if (b.p) {
        VS_CUDA(cudaStreamSynchronize(c->stream));
        VS_CUDA(cudaFree(b.p));
        b.p = nullptr;
        b.cap = 0;
    }
    size_t want = bytes < 256 ? 256 : bytes;
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) {
        b.p = nullptr;
        (void)cudaGetLastError();
        set_error("cudaMalloc of %zu bytes failed: %s", want, cudaGetErrorString(e));
        return VS_ERR_NOMEM;
    }
    b.cap = want;
    return VS_OK;
}

int stage_in(vs_ctx *c, DevBuf &scratch, const void *p, int mem, size_t bytes, const void **dev) {
    if (mem == VS_MEM_DEVICE) {
        *dev = p;
        return VS_OK;
    }
    VS_REQUIRE(mem == VS_MEM_HOST, VS_ERR_ARG, "bad memory flag %d", mem);
    VS_TRY(ensure(c, scratch, bytes));
    VS_CUDA(cudaMemcpyAsync(scratch.p, p, bytes, cudaMemcpyHostToDevice, c->stream));
    *dev = scratch.p;
    return VS_OK;
}

static int env_int(const char *name, int dflt) {
    const char *v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}

void load_options(Options &o) {
    o = Options();
    o.fused_variant = env_int("VS_FUSED_VARIANT", 0);
    o.no_pipeline = env_int("VS_NO_PIPELINE", 0);
    if (const char *t = getenv("VS_TRACE")) o.trace = t;
    o.gram_mma = env_int("VS_GRAM_MMA", -1);
    o.gram_mma_gen = env_int("VS_GRAM_GEN", -1);
    o.export_slow_gen = env_int("VS_EXPORT_SLOW_GEN", 0);
    o.export_copies = env_int("VS_EXPORT_COPIES", 0);
    o.gram_st = env_int("VS_GRAM_ST", 0);
    o.gram_warps = env_int("VS_GRAM_WARPS", 0);
    o.pf_rows = env_int("VS_PF_ROWS", 0);
    o.gram_rc = env_int("VS_GRAM_RC", 0);
    o.gram_stages = env_int("VS_GRAM_STAGES", 0);
    o.gram_debug = env_int("VS_GRAM_DEBUG", 0);
    o.p2p_timeout_ms = env_int("VS_P2P_TIMEOUT_MS", 10000);
    o.halton_mode = env_int("VS_HALTON_MODE", 0);
    o.index_bits = env_int("VS_INDEX_BITS", 0);
    o.no_bulk_export = env_int("VS_NO_BULK_EXPORT", 0);
    o.no_pf_eval = env_int("VS_NO_PF_EVAL", 0);
}

// Mapped pinned host memory the tail of the fused kernel writes its results to (no device-to-host copy call on the step).
int ensure_host_res(vs_ctx *c, size_t doubles) {
    if (c->host_res && c->host_res_cap >= doubles) return VS_OK;
    if (c->host_res) {
        VS_CUDA(cudaStreamSynchronize(c->stream));
        VS_CUDA(cudaFreeHost(c->host_res));
        c->host_res = nullptr;
        c->host_res_cap = 0;
    }
    size_t want = doubles < 4096 ? 4096 : doubles;
    VS_CUDA(cudaHostAlloc((void **)&c->host_res, want * sizeof(double), cudaHostAllocMapped | cudaHostAllocPortable));
    memset(c->host_res, 0, want * sizeof(double));
    c->host_res_cap = want;
    return VS_OK;
}

bool capturing(vs_ctx *c) {
    cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(c->stream, &st) != cudaSuccess) { (void)cudaGetLastError(); return false; }
    return st != cudaStreamCaptureStatusNone;
}
void time_begin(vs_ctx *c) {
    if (!c->timing || capturing(c)) return;       // events recorded inside a CUDA graph capture cannot be timed
    cudaEventRecord(c->ev0, c->stream);
}
void time_end(vs_ctx *c) {
    if (!c->timing || capturing(c)) return;
    cudaEventRecord(c->ev1, c->stream);
    c->timed = true;
}

// ---------------------------------------------------------------------------------------------
// Halton bases and term table
// ---------------------------------------------------------------------------------------------
static void first_primes(int k, std::vector<uint32_t> &p) {
    p.clear();
    for (uint32_t v = 2; (int)p.size() < k; ++v) {
        bool prime = true;
        for (size_t i = 0; i < p.size() && (uint64_t)p[i] * p[i] <= v; ++i)
            if (v % p[i] == 0) { prime = false; break; }
        if (prime) p.push_back(v);
    }
}

static void digit_counts(const std::vector<uint32_t> &bases, uint64_t max_index, std::vector<uint32_t> &nd) {
    nd.resize(bases.size());
    for (size_t d = 0; d < bases.size(); ++d) {
        uint32_t c = 0;
        for (uint64_t m = max_index; m > 0; m /= bases[d]) ++c;
        nd[d] = c ? c : 1;
    }
}

// The one place that fixes the generator's fp64 arithmetic (enum vs_halton_mode, include/varsens_b200.h).  Default: term =
// (double)digit / (double)b^(j+1), with b^(j+1) accumulated as ghalton does (bp *= b; exact for every index range we
// accept).  The kernels only add table entries in digit order, so re-pointing them at a different ghalton build -- should a
// real install ever disagree with the restatement, tests/golden/make_ghalton_golden.py -- is choosing another mode here.
static void build_terms(const std::vector<uint32_t> &bases, const std::vector<uint32_t> &nd, int mode, std::vector<uint32_t> &off,
                        std::vector<double> &terms) {
    off.resize(bases.size());
    terms.clear();
    for (size_t d = 0; d < bases.size(); ++d) {
        off[d] = (uint32_t)terms.size();
        volatile double bp = (double)bases[d];
        volatile double ib = 1.0 / (double)bases[d];
        volatile double f = ib;                                   // RUNNING_RECIPROCAL: f_j
        for (uint32_t j = 0; j < nd[d]; ++j) {
            volatile double rbp = 1.0 / bp;                       // RECIPROCAL: 1 / b^(j+1)
            for (uint32_t digit = 0; digit < bases[d]; ++digit) {
                volatile double q;
                if (mode == VS_HALTON_RECIPROCAL) q = (double)digit * rbp;
                else if (mode == VS_HALTON_RUNNING_RECIPROCAL) q = (double)digit * f;
                else q = (double)digit / bp;
                terms.push_back((double)q);
            }
            bp = bp * (double)bases[d];
            f = f * ib;
        }
    }
}

// Constants of the computed-term form (fused_impl.cuh: digit_step_arith) for every (dimension, digit position) a 32-bit
// index can reach, [k][HL_J]: term(digit) = fma(dd, rh, dd * rl) with dd = 8 * digit.  Returns whether they reproduce the
// term-table arithmetic of `mode` bit for bit, for every digit of every position (exhaustive).
static bool build_arith(const std::vector<uint32_t> &bases, int mode, std::vector<double> &arh, std::vector<double> &arl) {
    arh.assign(bases.size() * HL_J, 0.0);
    arl.assign(bases.size() * HL_J, 0.0);
    bool ok = true;
    for (size_t d = 0; d < bases.size(); ++d) {
        volatile double bp = (double)bases[d];
        volatile double ib = 1.0 / (double)bases[d];
        volatile double f = ib;
        for (int j = 0; j < HL_J; ++j) {
            if ((double)bp > 4294967296.0 * (double)bases[d]) break;     // position not reachable by a 32-bit index
            double rh, rl;
            if (mode == VS_HALTON_RECIPROCAL) { rh = 1.0 / bp; rl = 0.0; }
            else if (mode == VS_HALTON_RUNNING_RECIPROCAL) { rh = f; rl = 0.0; }
            else { rh = 1.0 / bp; rl = std::fma(-rh, (double)bp, 1.0) / bp; }
            arh[d * HL_J + j] = rh * 0.125;
            arl[d * HL_J + j] = rl * 0.125;
            for (uint32_t digit = 0; digit < bases[d]; ++digit) {
                volatile double want;
                if (mode == VS_HALTON_RECIPROCAL) want = (double)digit * (1.0 / bp);
                else if (mode == VS_HALTON_RUNNING_RECIPROCAL) want = (double)digit * f;
                else want = (double)digit / bp;
                const double dd = 8.0 * (double)digit;
                volatile double t = dd * arl[d * HL_J + j];
                const double got = std::fma(dd, arh[d * HL_J + j], (double)t);
                if (got != (double)want) ok = false;
            }
            bp = bp * (double)bases[d];
            f = f * ib;
        }
    }
    return ok;
}

int get_halton(vs_ctx *c, int k, uint64_t max_index, HaltonDev *out) {
    VS_REQUIRE(max_index < (1ull << 32), VS_ERR_RANGE, "Halton index %llu does not fit 32 bits",
               (unsigned long long)max_index);
    std::vector<uint32_t> bases, nd;
    first_primes(k, bases);
    digit_counts(bases, max_index, nd);
    HaltonCache &hc = c->halton;
    const int mode = c->opt.halton_mode;
    bool hit = hc.blob && hc.k == k && hc.mode == mode && hc.ndigits.size() == nd.size();
    if (hit)
        for (size_t d = 0; d < nd.size(); ++d)
            if (hc.ndigits[d] < nd[d]) { hit = false; break; }
    if (!hit) {
        std::vector<uint32_t> off;
        std::vector<double> terms;
        build_terms(bases, nd, mode == VS_HALTON_HORNER ? VS_HALTON_DIVIDE : mode, off, terms);
        std::vector<uint64_t> magic(k);
        for (int d = 0; d < k; ++d) magic[d] = (~0ull) / bases[d] + 1ull;   // floor((2^64-1)/b)+1 == floor(2^64/b)+1 for b not a power of 2; b=2 unused
        // The fused kernels keep the table in shared memory in a FIXED layout (fused_impl.cuh: foff / ndmax32): dimension d >= 1
        // owns ndmax32(b_d) rows -- every digit position a 32-bit index can have -- so that row addresses are compile-time
        // constants; it is built here once and copied by every CTA with one flat, coalesced loop.
        std::vector<double> fixed;
        if (k <= 32) {
            std::vector<uint32_t> nd32, off32;
            digit_counts(bases, 0xFFFFFFFFull, nd32);
            std::vector<uint32_t> b1(bases.begin() + 1, bases.end()), n1(nd32.begin() + 1, nd32.end());
            build_terms(b1, n1, mode == VS_HALTON_HORNER ? VS_HALTON_DIVIDE : mode, off32, fixed);
        }
        size_t nb_terms = terms.size() * sizeof(double), nb_magic = (size_t)k * 8, nb_u32 = (size_t)k * 4;
        size_t nb_fixed = ((fixed.size() + 1) & ~(size_t)1) * sizeof(double);
        nb_terms = (nb_terms + 15) & ~(size_t)15;
        std::vector<double> arh_h, arl_h;
        const bool arith_ok = build_arith(bases, mode == VS_HALTON_HORNER ? VS_HALTON_DIVIDE : mode, arh_h, arl_h);
        const size_t nb_ar = arh_h.size() * sizeof(double);
        size_t total = nb_terms + nb_fixed + 2 * nb_ar + nb_magic + 2 * nb_u32 + 64;
        if (hc.blob) {
            VS_CUDA(cudaStreamSynchronize(c->stream));
            VS_CUDA(cudaFree(hc.blob));
            hc.blob = nullptr;
        }
        VS_CUDA(cudaMalloc(&hc.blob, total));
        char *p = (char *)hc.blob;
        VS_CUDA(cudaMemcpy(p, terms.data(), terms.size() * sizeof(double), cudaMemcpyHostToDevice));
        hc.dev.terms = (const double *)p;
        p += nb_terms;
        if (!fixed.empty()) VS_CUDA(cudaMemcpy(p, fixed.data(), fixed.size() * sizeof(double), cudaMemcpyHostToDevice));
        hc.dev.fixed = fixed.empty() ? nullptr : (const double *)p;
        hc.dev.fixed_len = (uint32_t)fixed.size();
        p += nb_fixed;
        VS_CUDA(cudaMemcpy(p, arh_h.data(), nb_ar, cudaMemcpyHostToDevice));
        hc.dev.arh = (const double *)p;
        p += nb_ar;
        VS_CUDA(cudaMemcpy(p, arl_h.data(), nb_ar, cudaMemcpyHostToDevice));
        hc.dev.arl = (const double *)p;
        p += nb_ar;
        hc.dev.arith_ok = arith_ok ? 1 : 0;
        VS_CUDA(cudaMemcpy(p, magic.data(), nb_magic, cudaMemcpyHostToDevice));
        hc.dev.magic = (const uint64_t *)p;
        p += nb_magic;
        VS_CUDA(cudaMemcpy(p, bases.data(), nb_u32, cudaMemcpyHostToDevice));
        hc.dev.base = (const uint32_t *)p;
        p += nb_u32;
        VS_CUDA(cudaMemcpy(p, off.data(), nb_u32, cudaMemcpyHostToDevice));
        hc.dev.off = (const uint32_t *)p;
        hc.dev.total_terms = (uint32_t)terms.size();
        hc.k = k;
        hc.mode = mode;
        hc.ndigits = nd;
        hc.off = off;
        hc.arh = arh_h;
        hc.arl = arl_h;
        hc.arith_ok = arith_ok;
    }
    hc.dev.mode = mode;
    *out = hc.dev;
    return VS_OK;
}

int get_scale(vs_ctx *c, int k, const vs_scale *s, ScaleDev *out) {
    out->kind = VS_SCALE_IDENTITY;
    out->lb = out->wr = out->host = nullptr;
    if (!s || s->kind == VS_SCALE_IDENTITY) return VS_OK;
    VS_REQUIRE(s->kind == VS_SCALE_LINEAR || s->kind == VS_SCALE_POWER, VS_ERR_ARG, "unknown scale kind %d", s->kind);
    VS_REQUIRE(s->lower && s->upper, VS_ERR_ARG, "scale bounds are NULL");
    std::vector<double> h(2 * (size_t)k);
    for (int d = 0; d < k; ++d) {
        volatile double lo = s->lower[d], up = s->upper[d];
        volatile double wr = (s->kind == VS_SCALE_LINEAR) ? (up - lo) : (up / lo);   // scale.py:33 / :62
        h[d] = lo;
        h[k + d] = wr;
    }
    if (!(c->scale_kind_cached == s->kind && c->scale_k_cached == k && c->scale_host == h && c->scale_buf.p)) {
        VS_CUDA(cudaStreamSynchronize(c->stream));   // a kernel in flight may still read the old descriptor
        c->scale_host = h;
        VS_TRY(ensure(c, c->scale_buf, h.size() * sizeof(double)));
        VS_CUDA(cudaMemcpyAsync(c->scale_buf.p, c->scale_host.data(), h.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        c->scale_kind_cached = s->kind;
        c->scale_k_cached = k;
    }
    out->kind = s->kind;
    out->lb = (const double *)c->scale_buf.p;
    out->wr = out->lb + k;
    out->host = c->scale_host.data();
    return VS_OK;
}

int objective_host(int k, int objective, const double *params, int n_params, std::vector<double> *hp, int *l) {
    std::vector<double> scratch;
    std::vector<double> &h = hp ? *hp : scratch;
    *l = 1;
    switch (objective) {
    case VS_OBJ_GFUNCTION:
        VS_REQUIRE(params && n_params == k, VS_ERR_ARG, "g-function needs k=%d parameters a_c, got %d", k, n_params);
        h.resize(3 * (size_t)k);
        for (int d = 0; d < k; ++d) {
            VS_REQUIRE(params[d] > -1.0, VS_ERR_ARG, "g-function needs a_c > -1");
            h[d] = params[d];
            h[k + d] = 1.0 / (1.0 + params[d]);
            h[2 * k + d] = params[d] / (1.0 + params[d]);
        }
        break;
    case VS_OBJ_ISHIGAMI:
        VS_REQUIRE(k >= 3, VS_ERR_ARG, "Ishigami needs k >= 3");
        VS_REQUIRE(params && n_params == 2, VS_ERR_ARG, "Ishigami needs parameters {A, B}");
        h.assign(params, params + 2);
        break;
    case VS_OBJ_RK4_CHAIN:
        VS_REQUIRE(k >= 2 && k % 2 == 0 && k / 2 <= 64, VS_ERR_ARG, "RK4 chain needs even k with k/2 <= 64 links");
        VS_REQUIRE(params && n_params == 2 && params[1] >= 0, VS_ERR_ARG, "RK4 chain needs parameters {dt, nsteps}");
        h.assign(params, params + 2);
        break;
    case VS_OBJ_MASS_ACTION:
    case VS_OBJ_MASS_ACTION_ADAPTIVE:
    case VS_OBJ_MASS_ACTION_STIFF:
        return network_describe(k, objective, params, n_params, hp, l);
    default:
        set_error("unknown objective id %d", objective);
        return VS_ERR_ARG;
    }
    return VS_OK;
}

int get_objective(vs_ctx *c, int k, int objective, const double *params, int n_params, ObjectiveDev *out) {
    std::vector<double> h;
    int l = 1;
    VS_TRY(objective_host(k, objective, params, n_params, &h, &l));
    if (!(c->obj_id_cached == objective && c->obj_host == h && c->obj_buf.p)) {
        VS_CUDA(cudaStreamSynchronize(c->stream));   // a kernel in flight may still read the old parameters
        c->obj_host = h;
        VS_TRY(ensure(c, c->obj_buf, h.size() * sizeof(double)));
        VS_CUDA(cudaMemcpyAsync(c->obj_buf.p, c->obj_host.data(), h.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        c->obj_id_cached = objective;
    }
    out->id = objective;
    out->l = l;
    out->params = (const double *)c->obj_buf.p;
    out->n_params = (int)h.size();
    out->host = c->obj_host.data();
    return VS_OK;
}

int make_source(vs_ctx *c, int k, uint64_t n, uint64_t discard, const uint32_t *perm, int perm_mem, uint64_t perm_begin,
                uint64_t perm_count, const double *raw, int raw_mem, SourceDev *out) {
    memset(out, 0, sizeof(*out));
    VS_REQUIRE(perm, VS_ERR_ARG, "perm is NULL");
    // Both bounds hold before anything is added, so start + 2n - 1 below cannot wrap around 2^64 (a wrapped start would
    // reach Halton index 0, which is not a point of the sequence).
    VS_REQUIRE(discard < (1ull << 32) && n < (1ull << 32), VS_ERR_RANGE, "discard %llu or n %llu does not fit 32 bits",
               (unsigned long long)discard, (unsigned long long)n);
    out->n = n;
    out->start = 20ull * (uint64_t)k + discard + 1ull;          // saltelli.py:83: 20k + discard points skipped
    if (raw) {
        const void *d = nullptr;
        VS_TRY(stage_in(c, c->raw_buf, raw, raw_mem, 2 * n * (uint64_t)k * sizeof(double), &d));
        out->raw = (const double *)d;
    } else {
        uint64_t last = out->start + 2 * n - 1;
        VS_TRY(get_halton(c, k, last, &out->h));
    }
    // perm is indexed by the absolute base row i; stage only the slice a shard needs.
    const void *d = nullptr;
    if (perm_mem == VS_MEM_DEVICE) {
        out->perm = perm;
    } else {
        VS_TRY(stage_in(c, c->perm_buf, perm + perm_begin, VS_MEM_HOST, perm_count * sizeof(uint32_t), &d));
        out->perm = (const uint32_t *)d - perm_begin;
    }
    return VS_OK;
}

}  // namespace vs

// ---------------------------------------------------------------------------------------------
// extern "C": library / context / host helpers
// ---------------------------------------------------------------------------------------------
using namespace vs;

extern "C" int vs_abi_version(void) { return VS_ABI_VERSION; }

extern "C" int vs_objective_outputs(int k, int objective, const double *params, int n_params, int *l) {
    VS_REQUIRE(l, VS_ERR_ARG, "l is NULL");
    VS_REQUIRE(k >= 1 && k <= 4096, VS_ERR_ARG, "k=%d out of range [1,4096]", k);
    return objective_host(k, objective, params, n_params, nullptr, l);
}

extern "C" const char *vs_last_error(void) { return g_err; }

extern "C" int vs_ctx_create(int device, vs_ctx **out) {
    VS_REQUIRE(out, VS_ERR_ARG, "out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        (void)cudaGetLastError();
        set_error("no CUDA device available (%s); varsens_b200 has no CPU fallback",
                  e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        return VS_ERR_CUDA;
    }
    VS_REQUIRE(device >= 0 && device < count, VS_ERR_ARG, "device %d out of range [0,%d)", device, count);
    VS_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    VS_CUDA(cudaGetDeviceProperties(&prop, device));
    VS_REQUIRE(prop.major >= 10, VS_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a only",
               device, prop.major, prop.minor);
    vs_ctx *c = new vs_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->smem_optin = prop.sharedMemPerBlockOptin;
    VS_CUDA(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
    VS_CUDA(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    c->stream = c->own_stream;
    VS_CUDA(cudaEventCreate(&c->ev0));
    VS_CUDA(cudaEventCreate(&c->ev1));
    load_options(c->opt);
    *out = c;
    return VS_OK;
}

extern "C" int vs_ctx_destroy(vs_ctx *c) {
    if (!c) return VS_OK;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    cudaStreamSynchronize(c->copy_stream);
    if (c->host_res) cudaFreeHost(c->host_res);
    DevBuf *bufs[] = {&c->poll_buf, &c->ticket_buf, &c->peer_buf, &c->pipe_buf, &c->scale_buf, &c->obj_buf, &c->perm_buf, &c->raw_buf, &c->io_buf,
                      &c->part_buf,  &c->block_buf, &c->res_buf, &c->dir_buf, &c->misc_buf, &c->stats_buf};
    for (DevBuf *b : bufs)
        if (b->p) cudaFree(b->p);
    if (c->halton.blob) cudaFree(c->halton.blob);
    for (cudaEvent_t e : c->pipe_ev) cudaEventDestroy(e);
    cudaEventDestroy(c->ev0);
    cudaEventDestroy(c->ev1);
    cudaStreamDestroy(c->own_stream);
    cudaStreamDestroy(c->copy_stream);
    delete c;
    return VS_OK;
}

extern "C" int vs_ctx_set_stream(vs_ctx *c, void *stream) {
    VS_REQUIRE(c, VS_ERR_ARG, "ctx is NULL");
    VS_CUDA(cudaSetDevice(c->device));
    VS_CUDA(cudaStreamSynchronize(c->stream));
    c->stream = stream ? (cudaStream_t)stream : c->own_stream;
    return VS_OK;
}

extern "C" int vs_ctx_set_timing(vs_ctx *c, int on) {
    VS_REQUIRE(c, VS_ERR_ARG, "ctx is NULL");
    c->timing = on != 0;
    if (!c->timing) c->timed = false;
    return VS_OK;
}

extern "C" int vs_ctx_reload_env(vs_ctx *c) {
    VS_REQUIRE(c, VS_ERR_ARG, "ctx is NULL");
    load_options(c->opt);
    return VS_OK;
}

extern "C" int vs_ctx_synchronize(vs_ctx *c) {
    VS_REQUIRE(c, VS_ERR_ARG, "ctx is NULL");
    VS_CUDA(cudaSetDevice(c->device));
    VS_CUDA(cudaStreamSynchronize(c->stream));
    return VS_OK;
}

extern "C" uint64_t vs_ctx_launch_count(const vs_ctx *c) { return c ? c->launches : 0; }

extern "C" int vs_last_kernel_ms(vs_ctx *c, float *ms) {
    VS_REQUIRE(c && ms, VS_ERR_ARG, "NULL argument");
    VS_REQUIRE(c->timed, VS_ERR_ARG, "no timed kernel has run on this ctx (enable timing with vs_ctx_set_timing)");
    VS_CUDA(cudaSetDevice(c->device));
    VS_CUDA(cudaEventSynchronize(c->ev1));
    VS_CUDA(cudaEventElapsedTime(ms, c->ev0, c->ev1));
    return VS_OK;
}

extern "C" int vs_halton_bases(int k, uint32_t *bases) {
    VS_REQUIRE(k > 0 && bases, VS_ERR_ARG, "bad arguments");
    std::vector<uint32_t> b;
    first_primes(k, b);
    memcpy(bases, b.data(), sizeof(uint32_t) * k);
    return VS_OK;
}

extern "C" int vs_ctx_set_halton_mode(vs_ctx *c, int mode) {
    VS_REQUIRE(c, VS_ERR_ARG, "ctx is NULL");
    VS_REQUIRE(mode >= VS_HALTON_DIVIDE && mode <= VS_HALTON_HORNER, VS_ERR_ARG, "unknown Halton mode %d", mode);
    c->opt.halton_mode = mode;
    return VS_OK;
}

extern "C" int vs_halton_arith_check(int k, int mode) {
    if (k <= 0 || mode < VS_HALTON_DIVIDE || mode > VS_HALTON_RUNNING_RECIPROCAL) return -1;
    std::vector<uint32_t> bases;
    std::vector<double> arh, arl;
    first_primes(k, bases);
    return build_arith(bases, mode, arh, arl) ? 1 : 0;
}

extern "C" int vs_halton_terms(int k, uint64_t max_index, uint32_t *ndigits, uint32_t *offsets, double *terms,
                               uint64_t capacity, uint64_t *count) {
    return vs_halton_terms_mode(k, max_index, VS_HALTON_DIVIDE, ndigits, offsets, terms, capacity, count);
}

extern "C" int vs_halton_terms_mode(int k, uint64_t max_index, int mode, uint32_t *ndigits, uint32_t *offsets, double *terms,
                                    uint64_t capacity, uint64_t *count) {
    VS_REQUIRE(k > 0 && count, VS_ERR_ARG, "bad arguments");
    VS_REQUIRE(mode >= VS_HALTON_DIVIDE && mode <= VS_HALTON_RUNNING_RECIPROCAL, VS_ERR_UNSUPPORTED,
               "Halton mode %d has no term table", mode);
    std::vector<uint32_t> bases, nd, off;
    std::vector<double> t;
    first_primes(k, bases);
    digit_counts(bases, max_index, nd);
    build_terms(bases, nd, mode, off, t);
    *count = t.size();
    if (ndigits) memcpy(ndigits, nd.data(), sizeof(uint32_t) * k);
    if (offsets) memcpy(offsets, off.data(), sizeof(uint32_t) * k);
    if (terms) {
        VS_REQUIRE(capacity >= t.size(), VS_ERR_ARG, "terms capacity %llu < %zu", (unsigned long long)capacity, t.size());
        memcpy(terms, t.data(), sizeof(double) * t.size());
    }
    return VS_OK;
}

// ---------------------------------------------------------------------------------------------
// numpy.random.seed(s); numpy.random.shuffle(M_2)   (varsens/saltelli.py:100-101) as a row permutation.
// numpy's legacy global RNG is MT19937 seeded with init_genrand(s); shuffle walks i = n-1 .. 1 and swaps row i with row
// j = rk_interval(i): the smallest all-ones mask >= i, 32-bit draws AND-ed with it until the value is <= i.  The draws do
// not depend on the data, so they are produced a block ahead and the cache lines they will touch are prefetched -- the
// walk itself is a chain of random accesses into a 4n-byte array (64 MB at n = 2^24) and otherwise pays a full miss per
// swap.  key/pos give numpy's generator state AFTER the shuffle (the reference leaves the global RNG there).
// ---------------------------------------------------------------------------------------------
namespace {
struct MT19937 {
    uint32_t key[624];
    int pos;
    void seed(uint32_t s) {                                   // init_genrand (numpy: mt19937_seed)
        for (int i = 0; i < 624; ++i) {
            key[i] = s;
            s = 1812433253u * (s ^ (s >> 30)) + (uint32_t)i + 1u;
        }
        pos = 624;
    }
    void gen() {
        const uint32_t UPPER = 0x80000000u, LOWER = 0x7fffffffu, MATRIX_A = 0x9908b0dfu;
        int kk;
        uint32_t y;
        for (kk = 0; kk < 624 - 397; ++kk) {
            y = (key[kk] & UPPER) | (key[kk + 1] & LOWER);
            key[kk] = key[kk + 397] ^ (y >> 1) ^ (-(int32_t)(y & 1) & MATRIX_A);
        }
        for (; kk < 623; ++kk) {
            y = (key[kk] & UPPER) | (key[kk + 1] & LOWER);
            key[kk] = key[kk + (397 - 624)] ^ (y >> 1) ^ (-(int32_t)(y & 1) & MATRIX_A);
        }
        y = (key[623] & UPPER) | (key[0] & LOWER);
        key[623] = key[396] ^ (y >> 1) ^ (-(int32_t)(y & 1) & MATRIX_A);
        pos = 0;
    }
    inline uint32_t next() {
        if (pos == 624) gen();
        uint32_t y = key[pos++];
        y ^= (y >> 11);
        y ^= (y << 7) & 0x9d2c5680u;
        y ^= (y << 15) & 0xefc60000u;
        y ^= (y >> 18);
        return y;
    }
};
}  // namespace

extern "C" int vs_reference_permutation(uint64_t n, uint32_t seed, uint32_t *perm, uint32_t *key_out, int *pos_out) {
    VS_REQUIRE(perm || n == 0, VS_ERR_ARG, "perm is NULL");
    VS_REQUIRE(n <= 0xffffffffull, VS_ERR_RANGE, "n does not fit 32 bits");
    MT19937 mt;
    mt.seed(seed);
    for (uint64_t i = 0; i < n; ++i) perm[i] = (uint32_t)i;
    constexpr int AHEAD = 64;                                // draws produced (and lines prefetched) ahead of the swaps
    uint32_t js[AHEAD];
    uint64_t i = n > 0 ? n - 1 : 0;
    while (i >= 1) {
        const int cnt = (int)(i < (uint64_t)AHEAD ? i : (uint64_t)AHEAD);
        for (int u = 0; u < cnt; ++u) {
            const uint32_t mx = (uint32_t)(i - (uint64_t)u);
            uint32_t mask = mx;                               // smallest all-ones mask >= mx
            mask |= mask >> 1; mask |= mask >> 2; mask |= mask >> 4; mask |= mask >> 8; mask |= mask >> 16;
            uint32_t v;
            while ((v = (mt.next() & mask)) > mx) {}
            js[u] = v;
            __builtin_prefetch(perm + v, 1, 0);
        }
        for (int u = 0; u < cnt; ++u) {
            const uint64_t ii = i - (uint64_t)u;
            const uint32_t j = js[u], t = perm[ii];
            perm[ii] = perm[j];
            perm[j] = t;
        }
        i -= (uint64_t)cnt;
    }
    if (key_out) memcpy(key_out, mt.key, sizeof(mt.key));
    if (pos_out) *pos_out = mt.pos;
    return VS_OK;
}

extern "C" size_t vs_partials_len(int k, int l) {
    size_t m = (size_t)(2 + 2 * k) * (size_t)l;
    return 4 * (size_t)l + m * (m + 1) / 2;
}
