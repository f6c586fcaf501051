// extern "C" entry points (see include/varsens_b200.h for the contract of each).
#include <cstring>
#include <vector>

#include "vs_internal.cuh"

#include <cstdlib>

using namespace vs;

namespace {

// Output staging: run into `dev` (caller's device buffer or scratch), then copy to the host buffer.
struct OutStage {
    vs_ctx *c;
    void *user;
    int mem;
    size_t bytes;
    void *dev = nullptr;
    int begin(DevBuf &scratch) {
        if (mem == VS_MEM_DEVICE) {
            dev = user;
            return VS_OK;
        }
        VS_REQUIRE(mem == VS_MEM_HOST, VS_ERR_ARG, "bad memory flag %d", mem);
        VS_TRY(ensure(c, scratch, bytes));
        dev = scratch.p;
        return VS_OK;
    }
    int end() {
        if (mem == VS_MEM_HOST) {
            VS_CUDA(cudaMemcpyAsync(user, dev, bytes, cudaMemcpyDeviceToHost, c->stream));
            VS_CUDA(cudaStreamSynchronize(c->stream));
        }
        return VS_OK;
    }
};

int check_common(vs_ctx *c, int k) {
    VS_REQUIRE(c, VS_ERR_ARG, "ctx is NULL");
    VS_REQUIRE(k >= 1 && k <= 4096, VS_ERR_ARG, "k=%d out of range [1,4096]", k);
    VS_CUDA(cudaSetDevice(c->device));
    return VS_OK;
}

// Results the kernels write straight into the ctx's mapped host buffer (no copy call), in two steps around the launch.
// Before: a buffer large enough and a cleared status slot (finalize_kernel never writes it, so a time-out left by an earlier
// exchange cannot leak into a later call).
int host_result_begin(vs_ctx *c, int k, int l) {
    VS_TRY(ensure_host_res(c, result_len(k, l) + HOST_RES_EXTRA));
    c->host_res[result_len(k, l) + HOST_RES_STATUS] = 0.0;
    return VS_OK;
}

// After: wait for the kernel, fail on a peer time-out, copy out the fields the caller asked for.
int host_result_end(vs_ctx *c, int k, int l, int flags, vs_result *r) {
    VS_CUDA(cudaStreamSynchronize(c->stream));
    VS_REQUIRE(c->host_res[result_len(k, l) + HOST_RES_STATUS] == 0.0, VS_ERR_TIMEOUT,
               "peer-memory all-reduce: a rank did not publish its partial sums within %d ms", c->opt.p2p_timeout_ms);
    const double *p = c->host_res;
    const size_t kl = (size_t)k * l;
    auto take = [&](double *dst, size_t cnt) {
        if (dst) memcpy(dst, p, cnt * sizeof(double));
        p += cnt;
    };
    take(r->E_2, l);
    take(r->var_y, l);
    take(r->U_j, kl);
    take(r->U_nj, kl);
    take(r->sens, kl);
    take(r->sens_t, kl);
    if (flags & VS_FLAG_SECOND_ORDER) {
        take(r->sens_2, kl * kl);
        take(r->sens_2n, kl * kl);
    }
    return VS_OK;
}

// Estimators from partial sums in HBM.
int finalize_to_host(vs_ctx *c, int k, int l, uint64_t n, uint64_t rows, const double *partials_dev, int flags, vs_result *r) {
    VS_TRY(host_result_begin(c, k, l));
    VS_TRY(launch_finalize(c, k, l, n, rows, partials_dev, flags, c->host_res));
    return host_result_end(c, k, l, flags, r);
}

int check_estimator_args(int l, uint64_t n, uint64_t rows, bool pointers_set) {
    VS_REQUIRE(l >= 1 && l <= 64 && n >= 2 && rows >= 1 && rows <= n && pointers_set, VS_ERR_ARG, "bad arguments");
    return VS_OK;
}

// An all-device call only enqueues its work, but a host input it staged must have left the caller's buffer before it returns.
int sync_staged_inputs(vs_ctx *c, int out_mem, int perm_mem, const double *raw, int raw_mem) {
    if (out_mem == VS_MEM_DEVICE && (perm_mem == VS_MEM_HOST || (raw && raw_mem == VS_MEM_HOST)))
        VS_CUDA(cudaStreamSynchronize(c->stream));
    return VS_OK;
}

// The peer tables of an exchange as device arrays: every rank's buffer at [0, 64), its flag array at [64, 128) of peer_buf.
// Uploaded only when they change, once per exchange rather than once per step, after the work queued on the stream is done.
int peer_table(vs_ctx *c, int world_size, int rank, const uint64_t *peer_bufs, const uint64_t *peer_flags, uint32_t epoch,
               const uint64_t **tab) {
    VS_REQUIRE(world_size >= 1 && world_size <= 64 && rank >= 0 && rank < world_size && peer_bufs && epoch >= 1,
               VS_ERR_ARG, "bad peer description");
    VS_TRY(ensure(c, c->peer_buf, 2 * 64 * sizeof(uint64_t)));
    std::vector<uint64_t> want(128, 0);
    for (int r = 0; r < world_size; ++r) { want[r] = peer_bufs[r]; want[64 + r] = peer_flags ? peer_flags[r] : 0; }
    if (want != c->peer_tab) {
        VS_CUDA(cudaStreamSynchronize(c->stream));
        c->peer_tab = want;
        VS_CUDA(cudaMemcpyAsync(c->peer_buf.p, c->peer_tab.data(), 128 * sizeof(uint64_t), cudaMemcpyHostToDevice, c->stream));
    }
    *tab = (const uint64_t *)c->peer_buf.p;
    return VS_OK;
}

// Outputs per point of `objective`: 1 for every objective but a mass-action network, whose description is validated here.
int outputs_of(int k, int objective, const double *params, int n_params, int *l) {
    *l = 1;
    if (objective != VS_OBJ_MASS_ACTION && objective != VS_OBJ_MASS_ACTION_ADAPTIVE && objective != VS_OBJ_MASS_ACTION_STIFF)
        return VS_OK;
    return objective_host(k, objective, params, n_params, nullptr, l);
}

}  // namespace

extern "C" int vs_halton(vs_ctx *c, int k, uint64_t first_index, uint64_t count, const vs_scale *scale, double *out,
                         int out_mem) {
    VS_TRY(check_common(c, k));
    VS_REQUIRE(first_index >= 1, VS_ERR_ARG, "Halton indices are 1-based");
    if (count == 0) return VS_OK;
    VS_REQUIRE(out, VS_ERR_ARG, "out is NULL");
    HaltonDev h;
    VS_TRY(get_halton(c, k, first_index + count - 1, &h));
    ScaleDev s;
    VS_TRY(get_scale(c, k, scale, &s));
    OutStage o{c, out, out_mem, count * (uint64_t)k * sizeof(double)};
    VS_TRY(o.begin(c->io_buf));
    VS_TRY(launch_halton(c, k, first_index, count, h, s, (double *)o.dev));
    return o.end();
}

extern "C" int vs_sobol(vs_ctx *c, int k, uint64_t first_point, uint64_t count, const uint32_t *dirnums, int quantize6,
                        const vs_scale *scale, double *out, int out_mem) {
    VS_TRY(check_common(c, k));
    if (count == 0) return VS_OK;
    VS_REQUIRE(out && dirnums, VS_ERR_ARG, "NULL argument");
    VS_REQUIRE(first_point + count - 1 < (1ull << 32), VS_ERR_RANGE, "Sobol point number does not fit 32 bits");
    ScaleDev s;
    VS_TRY(get_scale(c, k, scale, &s));
    VS_TRY(ensure(c, c->dir_buf, (size_t)k * 32 * sizeof(uint32_t)));
    VS_CUDA(cudaMemcpyAsync(c->dir_buf.p, dirnums, (size_t)k * 32 * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
    OutStage o{c, out, out_mem, count * (uint64_t)k * sizeof(double)};
    VS_TRY(o.begin(c->io_buf));
    VS_TRY(launch_sobol(c, k, first_point, count, (const uint32_t *)c->dir_buf.p, quantize6, s, (double *)o.dev));
    VS_TRY(o.end());
    if (out_mem == VS_MEM_DEVICE) VS_CUDA(cudaStreamSynchronize(c->stream));   // dirnums is caller memory
    return VS_OK;
}

extern "C" int vs_sample_flat(vs_ctx *c, int k, uint64_t n, uint64_t discard, const uint32_t *perm, int perm_mem,
                              const double *raw, int raw_mem, const vs_scale *scale, uint64_t row_begin, uint64_t row_end,
                              double *out, int out_mem) {
    VS_TRY(check_common(c, k));
    VS_REQUIRE(n >= 1, VS_ERR_ARG, "n must be >= 1");
    uint64_t total = 2 * n * (1 + (uint64_t)k);
    VS_REQUIRE(row_begin <= row_end && row_end <= total, VS_ERR_ARG, "row window [%llu,%llu) outside [0,%llu)",
               (unsigned long long)row_begin, (unsigned long long)row_end, (unsigned long long)total);
    if (row_begin == row_end) return VS_OK;
    VS_REQUIRE(out, VS_ERR_ARG, "out is NULL");
    SourceDev src;
    VS_TRY(make_source(c, k, n, discard, perm, perm_mem, 0, n, raw, raw_mem, &src));
    ScaleDev s;
    VS_TRY(get_scale(c, k, scale, &s));
    OutStage o{c, out, out_mem, (row_end - row_begin) * (uint64_t)k * sizeof(double)};
    VS_TRY(o.begin(c->io_buf));
    VS_TRY(launch_sample_flat(c, k, src, s, row_begin, row_end, (double *)o.dev));
    VS_TRY(o.end());
    return sync_staged_inputs(c, out_mem, perm_mem, raw, raw_mem);
}

extern "C" int vs_sample_flat_shard(vs_ctx *c, int k, uint64_t n, uint64_t discard, const uint32_t *perm, int perm_mem,
                                    const double *raw, int raw_mem, const vs_scale *scale, uint64_t i_begin, uint64_t i_end,
                                    double *out, int out_mem) {
    VS_TRY(check_common(c, k));
    VS_REQUIRE(n >= 1 && i_begin <= i_end && i_end <= n, VS_ERR_ARG, "bad base-row range [%llu,%llu) of %llu",
               (unsigned long long)i_begin, (unsigned long long)i_end, (unsigned long long)n);
    if (i_begin == i_end) return VS_OK;
    VS_REQUIRE(out, VS_ERR_ARG, "out is NULL");
    SourceDev src;
    VS_TRY(make_source(c, k, n, discard, perm, perm_mem, i_begin, i_end - i_begin, raw, raw_mem, &src));
    ScaleDev s;
    VS_TRY(get_scale(c, k, scale, &s));
    OutStage o{c, out, out_mem, (i_end - i_begin) * (uint64_t)(2 + 2 * k) * (uint64_t)k * sizeof(double)};
    VS_TRY(o.begin(c->io_buf));
    VS_TRY(launch_sample_shard(c, k, src, s, i_begin, i_end, (double *)o.dev));
    VS_TRY(o.end());
    return sync_staged_inputs(c, out_mem, perm_mem, raw, raw_mem);
}

extern "C" int vs_eval_values(vs_ctx *c, int k, uint64_t n, uint64_t discard, const uint32_t *perm, int perm_mem,
                              const double *raw, int raw_mem, const vs_scale *scale, int objective, const double *params,
                              int n_params, uint64_t i_begin, uint64_t i_end, double *fvals, int fvals_mem) {
    VS_TRY(check_common(c, k));
    VS_REQUIRE(n >= 1 && i_begin <= i_end && i_end <= n, VS_ERR_ARG, "bad row range");
    if (i_begin == i_end) return VS_OK;
    VS_REQUIRE(fvals, VS_ERR_ARG, "fvals is NULL");
    SourceDev src;
    VS_TRY(make_source(c, k, n, discard, perm, perm_mem, i_begin, i_end - i_begin, raw, raw_mem, &src));
    ScaleDev s;
    VS_TRY(get_scale(c, k, scale, &s));
    ObjectiveDev od;
    VS_TRY(get_objective(c, k, objective, params, n_params, &od));
    OutStage o{c, fvals, fvals_mem, (i_end - i_begin) * (uint64_t)(2 + 2 * k) * od.l * sizeof(double)};
    VS_TRY(o.begin(c->io_buf));
    VS_TRY(launch_eval_values(c, k, src, s, od, i_begin, i_end, (double *)o.dev));
    VS_TRY(o.end());
    if (fvals_mem == VS_MEM_DEVICE) VS_CUDA(cudaStreamSynchronize(c->stream));
    return VS_OK;
}

extern "C" int vs_partials_from_values(vs_ctx *c, int k, int l, uint64_t rows, const double *fvals, int fvals_mem,
                                       const double *shift, int flags, double *partials, int partials_mem) {
    VS_TRY(check_common(c, k));
    VS_REQUIRE(l >= 1 && l <= 64, VS_ERR_ARG, "l=%d out of range [1,64]", l);
    VS_REQUIRE(partials && (fvals || rows == 0), VS_ERR_ARG, "NULL argument");
    size_t plen = vs_partials_len(k, l);
    OutStage o{c, partials, partials_mem, plen * sizeof(double)};
    VS_TRY(o.begin(c->part_buf));
    if (rows == 0) {
        VS_CUDA(cudaMemsetAsync(o.dev, 0, plen * sizeof(double), c->stream));
        return o.end();
    }
    const void *fdev = nullptr;
    VS_TRY(stage_in(c, c->io_buf, fvals, fvals_mem, rows * (uint64_t)(2 + 2 * k) * l * sizeof(double), &fdev));
    const double *shift_dev = nullptr;
    if (shift) {
        VS_TRY(ensure(c, c->misc_buf, 64 * sizeof(double)));
        VS_CUDA(cudaMemcpyAsync(c->misc_buf.p, shift, l * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        shift_dev = (const double *)c->misc_buf.p;
    }
    VS_TRY(launch_partials_from_values(c, k, l, rows, (const double *)fdev, shift_dev, flags, (double *)o.dev));
    VS_TRY(o.end());
    if (partials_mem == VS_MEM_DEVICE) VS_CUDA(cudaStreamSynchronize(c->stream));
    return VS_OK;
}

extern "C" int vs_finalize(vs_ctx *c, int k, int l, uint64_t n, uint64_t rows, const double *partials, int partials_mem,
                           int flags, vs_result *result) {
    VS_TRY(check_common(c, k));
    VS_TRY(check_estimator_args(l, n, rows, partials && result));
    const void *pdev = nullptr;
    VS_TRY(stage_in(c, c->part_buf, partials, partials_mem, vs_partials_len(k, l) * sizeof(double), &pdev));
    return finalize_to_host(c, k, l, n, rows, (const double *)pdev, flags, result);
}

extern "C" int vs_finalize_device(vs_ctx *c, int k, int l, uint64_t n, uint64_t rows, const double *partials_dev, int flags,
                                  double *result_dev) {
    VS_TRY(check_common(c, k));
    VS_TRY(check_estimator_args(l, n, rows, partials_dev && result_dev));
    return launch_finalize(c, k, l, n, rows, partials_dev, flags, result_dev);
}

extern "C" int vs_allreduce_finalize_p2p(vs_ctx *c, int k, int l, uint64_t n, uint64_t rows, int world_size, int rank,
                                         const uint64_t *peer_bufs, const uint64_t *peer_flags, uint32_t epoch,
                                         const double *partials_dev, int flags, vs_result *result) {
    VS_TRY(check_common(c, k));
    VS_TRY(check_estimator_args(l, n, rows, partials_dev && result));
    const uint64_t *tab = nullptr;
    VS_TRY(peer_table(c, world_size, rank, peer_bufs, peer_flags, epoch, &tab));
    VS_TRY(host_result_begin(c, k, l));
    VS_TRY(launch_p2p_reduce_finalize(c, k, l, n, rows, world_size, rank, tab, tab + 64, epoch, partials_dev, flags, c->host_res));
    return host_result_end(c, k, l, flags, result);
}

extern "C" int vs_indices_from_values(vs_ctx *c, int k, int l, uint64_t n, uint64_t rows, const double *fvals, int fvals_mem,
                                      int flags, vs_result *result) {
    VS_TRY(check_common(c, k));
    VS_TRY(check_estimator_args(l, n, rows, fvals && result));
    const void *fdev = nullptr;
    VS_TRY(stage_in(c, c->io_buf, fvals, fvals_mem, rows * (uint64_t)(2 + 2 * k) * l * sizeof(double), &fdev));
    // common shift = first row of fM_1 (any value works; this one is cheap and data-scaled)
    VS_TRY(ensure(c, c->misc_buf, 64 * sizeof(double)));
    VS_CUDA(cudaMemcpyAsync(c->misc_buf.p, fdev, l * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
    VS_TRY(ensure(c, c->part_buf, vs_partials_len(k, l) * sizeof(double)));
    VS_TRY(launch_partials_from_values(c, k, l, rows, (const double *)fdev, (const double *)c->misc_buf.p, flags,
                                       (double *)c->part_buf.p));
    return finalize_to_host(c, k, l, n, rows, (const double *)c->part_buf.p, flags, result);
}

// ---------------------------------------------------------------------------------------------------------------------
// The fused step.  One kernel launch does everything (fused_impl.cuh): generation + evaluation + Gram, fixed-order
// combine by the last CTA, and -- depending on FusedReq::mode -- the packed partial sums, the estimators, or the
// peer-memory all-reduce followed by the estimators, with the results written to mapped host memory.
//
// Host permutation (VS_MEM_HOST): the H2D copy (4 bytes per base row: 64 MB at n = 2^24, ~1.2 ms over PCIe) is ONE
// cudaMemcpyAsync on the copy stream into a staging buffer whose entries hold a sentinel; the SAME single launch runs while the
// bytes arrive -- every lane polls its own entry -- so only the first few hundred KB are exposed and no launch is repeated.
// The copy is enqueued before the launch (a serialising tool -- compute-sanitizer, CUDA_LAUNCH_BLOCKING -- cannot deadlock).
// ---------------------------------------------------------------------------------------------------------------------
static const uint64_t PIPE_MIN_ROWS = 1ull << 19;

static int fused_step(vs_ctx *c, int k, uint64_t n, uint64_t discard, const uint32_t *perm, int perm_mem, const double *raw,
                      int raw_mem, const vs_scale *scale, int objective, const double *params, int n_params, uint64_t i_begin,
                      uint64_t i_end, int flags, double *partials_dev, FusedReq *req, bool *finalized) {
    *finalized = false;
    const uint64_t rows = i_end - i_begin;
    const bool fused = fused_supported(k, objective, flags) && !(c->opt.halton_mode == VS_HALTON_HORNER && !raw);
    const bool tail_ok = fused && fused_tail_supported(c, k, objective, flags);
    ScaleDev s;
    ObjectiveDev od;
    SourceDev src;
    if (perm_mem == VS_MEM_HOST && !raw && tail_ok && rows >= PIPE_MIN_ROWS && !capturing(c) && !c->opt.no_pipeline) {
        VS_REQUIRE(perm, VS_ERR_ARG, "perm is NULL");
        // Staging buffer whose entries hold the sentinel 0xFFFFFFFF between calls: ONE asynchronous copy is enqueued (before the
        // launch, so a serialising tool cannot deadlock), the kernel's lanes poll their own entries and put the sentinel back.
        if (c->poll_buf.cap < rows * sizeof(uint32_t) || !c->poll_clean) {
            VS_TRY(ensure(c, c->poll_buf, rows * sizeof(uint32_t)));
            VS_CUDA(cudaMemsetAsync(c->poll_buf.p, 0xFF, c->poll_buf.cap, c->stream));
        }
        c->poll_clean = false;                                                  // until the launch below is enqueued
        if (c->pipe_ev.empty()) {
            cudaEvent_t e;
            VS_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            c->pipe_ev.push_back(e);
        }
        const uint32_t *perm_dev = (const uint32_t *)c->poll_buf.p - i_begin;      // indexed by the absolute base row
        VS_TRY(make_source(c, k, n, discard, perm_dev, VS_MEM_DEVICE, i_begin, rows, nullptr, VS_MEM_HOST, &src));
        VS_TRY(get_scale(c, k, scale, &s));
        VS_TRY(get_objective(c, k, objective, params, n_params, &od));
        // the copy may not start before earlier work on the compute stream (the previous kernel's sentinel stores, the refill)
        VS_CUDA(cudaEventRecord(c->pipe_ev[0], c->stream));
        VS_CUDA(cudaStreamWaitEvent(c->copy_stream, c->pipe_ev[0], 0));
        VS_CUDA(cudaMemcpyAsync(c->poll_buf.p, perm + i_begin, rows * sizeof(uint32_t), cudaMemcpyHostToDevice, c->copy_stream));
        req->poll_perm = 1;
        VS_TRY(launch_fused(c, k, src, s, od, i_begin, i_end, flags, partials_dev, req, finalized));
        c->poll_clean = true;                                                   // the kernel leaves every entry it read at the sentinel
        return VS_OK;
    }
    VS_TRY(make_source(c, k, n, discard, perm, perm_mem, i_begin, rows, raw, raw_mem, &src));
    VS_TRY(get_scale(c, k, scale, &s));
    VS_TRY(get_objective(c, k, objective, params, n_params, &od));
    if (fused) {
        if (!tail_ok || capturing(c)) {                  // legacy variants (and graph capture) produce partial sums only
            FusedReq plain;
            if (!partials_dev) {
                VS_TRY(ensure(c, c->part_buf, vs_partials_len(k, 1) * sizeof(double)));
                partials_dev = (double *)c->part_buf.p;
            }
            return launch_fused(c, k, src, s, od, i_begin, i_end, flags, partials_dev, tail_ok ? &plain : nullptr, finalized);
        }
        return launch_fused(c, k, src, s, od, i_begin, i_end, flags, partials_dev, req, finalized);
    }
    // Two-phase path on the GPU: values to HBM scratch, then the Gram reduction.
    VS_REQUIRE(!(flags & VS_FLAG_SEPARABLE), VS_ERR_UNSUPPORTED, "VS_FLAG_SEPARABLE needs a fused kernel (objective %d, k=%d)",
               objective, k);
    VS_REQUIRE(partials_dev, VS_ERR_ARG, "two-phase path needs a partial-sum buffer");
    const int l = od.l;                              // values laid out fvals[(t*rows + r)*l + o]
    VS_TRY(ensure(c, c->io_buf, rows * (uint64_t)(2 + 2 * k) * l * sizeof(double)));
    VS_TRY(launch_eval_values(c, k, src, s, od, i_begin, i_end, (double *)c->io_buf.p));
    // common shift: the l values of f(M_1[0]), which must not depend on the shard: evaluate base row 0 separately
    VS_TRY(ensure(c, c->misc_buf, (size_t)(64 + (2 + 2 * k) * l) * sizeof(double)));
    if (i_begin == 0) {
        VS_CUDA(cudaMemcpyAsync(c->misc_buf.p, c->io_buf.p, l * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
    } else {
        SourceDev src0 = src;
        if (perm_mem == VS_MEM_HOST) {   // row 0's permutation entry is outside the staged slice
            VS_TRY(ensure(c, c->dir_buf, 256));
            VS_CUDA(cudaMemcpyAsync(c->dir_buf.p, perm, sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
            src0.perm = (const uint32_t *)c->dir_buf.p;
        }
        double *tmp = (double *)c->misc_buf.p + 64;
        VS_TRY(launch_eval_values(c, k, src0, s, od, 0, 1, tmp, false));   // not part of the shard's step counts
        VS_CUDA(cudaMemcpyAsync(c->misc_buf.p, tmp, l * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
    }
    return launch_partials_from_values(c, k, l, rows, (const double *)c->io_buf.p, (const double *)c->misc_buf.p, flags,
                                       partials_dev);
}

extern "C" int vs_fused_partials(vs_ctx *c, int k, uint64_t n, uint64_t discard, const uint32_t *perm, int perm_mem,
                                 const double *raw, int raw_mem, const vs_scale *scale, int objective, const double *params,
                                 int n_params, uint64_t i_begin, uint64_t i_end, int flags, double *partials, int partials_mem) {
    VS_TRY(check_common(c, k));
    VS_REQUIRE(n >= 2 && i_begin <= i_end && i_end <= n && partials, VS_ERR_ARG, "bad arguments");
    int l = 1;
    VS_TRY(outputs_of(k, objective, params, n_params, &l));
    size_t plen = vs_partials_len(k, l);
    OutStage o{c, partials, partials_mem, plen * sizeof(double)};
    VS_TRY(o.begin(c->part_buf));
    if (i_begin == i_end) {
        VS_CUDA(cudaMemsetAsync(o.dev, 0, plen * sizeof(double), c->stream));
        return o.end();
    }
    FusedReq req;
    bool finalized = false;
    VS_TRY(fused_step(c, k, n, discard, perm, perm_mem, raw, raw_mem, scale, objective, params, n_params, i_begin, i_end, flags,
                      (double *)o.dev, &req, &finalized));
    VS_TRY(o.end());
    // all-device call: only enqueued (the caller's next op on the same stream, e.g. the all-reduce, orders after it)
    return sync_staged_inputs(c, partials_mem, perm_mem, raw, raw_mem);
}

extern "C" int vs_run_fused(vs_ctx *c, int k, uint64_t n, uint64_t discard, const uint32_t *perm, int perm_mem,
                            const double *raw, int raw_mem, const vs_scale *scale, int objective, const double *params,
                            int n_params, int flags, vs_result *result) {
    VS_TRY(check_common(c, k));
    VS_REQUIRE(n >= 2 && result, VS_ERR_ARG, "bad arguments");
    int l = 1;
    VS_TRY(outputs_of(k, objective, params, n_params, &l));
    VS_TRY(ensure(c, c->part_buf, vs_partials_len(k, l) * sizeof(double)));
    FusedReq req;
    req.mode = 1;
    req.n_total = req.rows_total = n;
    bool finalized = false;
    VS_TRY(host_result_begin(c, k, l));
    VS_TRY(fused_step(c, k, n, discard, perm, perm_mem, raw, raw_mem, scale, objective, params, n_params, 0, n, flags,
                      (double *)c->part_buf.p, &req, &finalized));
    if (!finalized) VS_TRY(launch_finalize(c, k, l, n, n, (const double *)c->part_buf.p, flags, c->host_res));
    return host_result_end(c, k, l, flags, result);
}

extern "C" int vs_run_fused_p2p(vs_ctx *c, int k, uint64_t n, uint64_t discard, const uint32_t *perm, int perm_mem,
                                const double *raw, int raw_mem, const vs_scale *scale, int objective, const double *params,
                                int n_params, uint64_t i_begin, uint64_t i_end, int flags, int world_size, int rank,
                                const uint64_t *peer_bufs, const uint64_t *peer_flags, uint32_t epoch, vs_result *result) {
    VS_TRY(check_common(c, k));
    VS_REQUIRE(n >= 2 && i_begin < i_end && i_end <= n && result, VS_ERR_ARG, "bad arguments (every rank needs at least one base row)");
    const uint64_t *tab = nullptr;
    VS_TRY(peer_table(c, world_size, rank, peer_bufs, peer_flags, epoch, &tab));
    int l = 1;
    VS_TRY(outputs_of(k, objective, params, n_params, &l));
    VS_TRY(ensure(c, c->part_buf, 2 * vs_partials_len(k, l) * sizeof(double)));
    double *mine = (double *)c->part_buf.p + vs_partials_len(k, l);       // [0, plen) is the scratch of the stand-alone exchange kernel
    FusedReq req;
    req.mode = 2;
    req.n_total = req.rows_total = n;
    req.world = world_size;
    req.rank = rank;
    req.epoch = epoch;
    req.peer_bufs_dev = tab;
    req.peer_flags_dev = tab + 64;
    bool finalized = false;
    VS_TRY(host_result_begin(c, k, l));
    VS_TRY(fused_step(c, k, n, discard, perm, perm_mem, raw, raw_mem, scale, objective, params, n_params, i_begin, i_end, flags,
                      mine, &req, &finalized));
    // kernels without the in-kernel tail (two-phase path, legacy variants): exchange + estimators in the stand-alone kernel
    if (!finalized)
        VS_TRY(launch_p2p_reduce_finalize(c, k, l, n, n, world_size, rank, tab, tab + 64, epoch, mine, flags, c->host_res));
    return host_result_end(c, k, l, flags, result);
}

extern "C" int vs_last_tail_ns(vs_ctx *c, int k, double *ns8) {
    VS_REQUIRE(c && ns8 && c->host_res, VS_ERR_ARG, "no fused step has run on this ctx");
    const double *x = c->host_res + result_len(k, 1) + HOST_RES_STAMPS;    // the fused kernel's tail has one output per point
    for (int i = 0; i < 11; ++i) ns8[i] = x[i];
    return VS_OK;
}

extern "C" int vs_last_network_stats(vs_ctx *c, uint64_t stats[4]) {
    VS_REQUIRE(c && stats, VS_ERR_ARG, "NULL argument");
    VS_REQUIRE(c->stats_buf.p, VS_ERR_ARG, "no adaptive or stiff mass-action network has been evaluated on this ctx");
    VS_CUDA(cudaSetDevice(c->device));
    VS_CUDA(cudaMemcpyAsync(stats, c->stats_buf.p, 4 * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
    VS_CUDA(cudaStreamSynchronize(c->stream));
    return VS_OK;
}

extern "C" int vs_measure_fp64_peak(vs_ctx *c, double *tflops) {
    VS_REQUIRE(c && tflops, VS_ERR_ARG, "NULL argument");
    VS_CUDA(cudaSetDevice(c->device));
    return launch_fp64_peak(c, tflops);
}
