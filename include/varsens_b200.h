/* varsens_b200 -- C ABI of the B200-native Saltelli hot path (libvarsens_b200.so).
 *
 * The reference (LoLab-MSM/varsens) has no FFI: its boundary is the Python API of
 * varsens/saltelli.py and varsens/scale.py.  Every entry point below names the reference code it
 * replaces (file:line under the reference checkout); varsens_b200/saltelli.py is the host mirror
 * that binds them through ctypes (INTEGRATION.md shows the stub a reference maintainer would add).
 *
 * Conventions
 *  - plain C symbols, int status return (VS_OK == 0), no exceptions cross the ABI;
 *    vs_last_error() returns the thread-local message of the last failing call.
 *  - the CALLER owns every data buffer.  Each buffer argument is paired with a VS_MEM_* flag:
 *    VS_MEM_DEVICE = device pointer on the ctx's GPU (e.g. torch.Tensor.data_ptr()),
 *    VS_MEM_HOST   = host pointer (numpy); the library stages it through its own device scratch
 *    with cudaMemcpyAsync on the ctx stream (pinned host memory makes that copy asynchronous).
 *  - small descriptor arguments (vs_scale bounds, objective parameters, direction numbers,
 *    vs_result arrays) are always HOST memory.
 *  - one in-flight call per ctx; calls are issued on the ctx stream and return after the stream
 *    has been synchronised unless the output is VS_MEM_DEVICE (then the work is only enqueued).
 *  - everything is IEEE fp64; indices are uint64 in the ABI (Halton index of any generated point
 *    must stay below 2^32: VS_ERR_RANGE otherwise).
 *  - there is NO CPU fallback: without a CUDA device vs_ctx_create fails with VS_ERR_CUDA.
 *  - limits (checked, never silent): 1 <= k <= 4096 for the generators, export mode and the estimators; vs_eval_values and
 *    the two-phase route of vs_fused_partials / vs_run_fused need the 2k coordinates of 32 rows in shared memory
 *    (k <= 453, VS_ERR_UNSUPPORTED beyond); the one-kernel fused route covers 2 <= k <= 20, other k take the two-phase
 *    route inside the same calls; 1 <= l <= 64 outputs per evaluation (VS_ERR_ARG beyond: the reference has no such limit,
 *    split the outputs into groups if the cross-output blocks of sens_2 are not needed).
 */
#ifndef VARSENS_B200_H
#define VARSENS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VS_ABI_VERSION 1

typedef struct vs_ctx vs_ctx;

enum vs_status { VS_OK = 0, VS_ERR_ARG = 1, VS_ERR_CUDA = 2, VS_ERR_RANGE = 3, VS_ERR_NOMEM = 4, VS_ERR_UNSUPPORTED = 5,
                 VS_ERR_TIMEOUT = 6 /* a peer rank did not show up in the peer-memory all-reduce */ };
enum vs_mem { VS_MEM_HOST = 0, VS_MEM_DEVICE = 1 };

/* varsens/scale.py: identity (lambda x: x), linear (:33), power (:62).  percentage (:90-91) lowers
 * to linear and magnitude (:121-122) to power on the host, exactly as scale.py does. */
enum vs_scale_kind { VS_SCALE_IDENTITY = 0, VS_SCALE_LINEAR = 1, VS_SCALE_POWER = 2 };
typedef struct vs_scale {
    int kind;
    const double *lower; /* host, k doubles (ignored for identity) */
    const double *upper; /* host, k doubles */
} vs_scale;

/* Registered device objective functors (the reference calls a Python callable once per row,
 * varsens/saltelli.py:308-353).  params are host doubles:
 *   GFUNCTION  : a[0..k)                      f = prod_c (|4 x_c - 2| + a_c) / (1 + a_c)
 *                (varsens/tests/test_g_function.py:9-13, README.md:33-36)
 *   ISHIGAMI   : {A, B}, k >= 3               f = sin x0 + A sin^2 x1 + B x2^4 sin x0
 *   RK4_CHAIN  : {dt, nsteps}, k even         reversible mass-action chain X_0 <-> ... <-> X_{k/2},
 *                forward rates x[0..k/2), reverse rates x[k/2..k), X(0) = e_0, classic RK4,
 *                f = X_{k/2}(nsteps*dt)       (spec frozen in oracle/objectives.py)
 *   MASS_ACTION: a run-time mass-action reaction network integrated by classic fixed-step RK4, L observables
 *                (l = L outputs per point).  params, indices stored as exact integers, -1 = none / use the constant:
 *                  [0] S  [1] R  [2] L  [3] dt  [4] nsteps
 *                  R records of 8:  a0 a1 b0 b1  kf_coord kf_const  kr_coord kr_const
 *                                   (a = reactants, b = products: species index or -1; kr_coord = -1 with kr_const = 0
 *                                    is an irreversible reaction, its reverse term is not evaluated)
 *                  S records of 2:  init_coord init_const
 *                  L*S weights:     w[o][s]      observable o = sum_s w[o][s] X_s(nsteps*dt), zero weights skipped
 *                n_params == 5 + 8R + 2S + L*S.  A rate or initial amount is x[coord] (the scaled sample coordinate,
 *                coord < k) when coord >= 0, else the constant.  Limits: 1 <= S <= 128, 1 <= R <= 512, 1 <= L <= 64,
 *                dt finite, 0 <= nsteps < 2^31, species indices < S, coordinates < k; anything else is VS_ERR_ARG.
 *                A network whose per-trajectory state does not fit the kernel's shared memory (k + 3S + R doubles per
 *                thread, 32 threads at least) is VS_ERR_UNSUPPORTED.  Two-phase route only; VS_FLAG_SEPARABLE is
 *                VS_ERR_UNSUPPORTED.  Frozen arithmetic (bit-identical to the oracle, and to RK4_CHAIN for the chain
 *                written as a network) in varsens_b200/csrc/device.cuh: MassAction.
 *   MASS_ACTION_ADAPTIVE: the same network integrated by adaptive Dormand-Prince 5(4) with error control, its L observables
 *                reported at NT output times (l = L*NT outputs per point).  Records, initial amounts and weights exactly as
 *                MASS_ACTION; only the header differs, and the output times follow the weights:
 *                  [0] S  [1] R  [2] L  [3] NT  [4] rtol  [5] atol  [6] h0  [7] max_steps
 *                  R records of 8, S records of 2, L*S weights
 *                  NT output times  0 < t_1 < t_2 < ... < t_NT   (integration starts at t = 0)
 *                n_params == 8 + 8R + 2S + L*S + NT; output column m*L + o = observable o at time t_{m+1}.  Limits: those of
 *                MASS_ACTION, 1 <= NT and L*NT <= 64, times finite and strictly increasing from > 0, rtol finite >= 0, atol
 *                finite > 0, h0 finite > 0, 1 <= max_steps < 2^31 (an integer); anything else is VS_ERR_ARG.  Each trajectory
 *                picks its own steps (error of a step against rtol*|X_s| + atol) and lands exactly on every output time.  A
 *                trajectory that needs more than max_steps attempts, or whose step no longer advances t, is failed: its
 *                outputs from the time it did not reach on are NaN (an ordinary value, see vs_last_network_stats).  State:
 *                k + 8S + R doubles per thread, 32 threads at least, else VS_ERR_UNSUPPORTED.  Two-phase route only;
 *                VS_FLAG_SEPARABLE is VS_ERR_UNSUPPORTED.  Frozen arithmetic in device.cuh: MassActionAdaptive.
 *   MASS_ACTION_STIFF: the same network and exactly the same params as MASS_ACTION_ADAPTIVE (header, records, initial
 *                amounts, weights, output times, l = L*NT, limits, output times and failure rules), integrated by the
 *                L-stable adaptive Rosenbrock method Rodas3 for stiff networks (rates many orders of magnitude apart).  One
 *                sparse Jacobian and LU factorisation per attempted step, in a fill-reducing order derived once per
 *                network; a zero or non-finite pivot rejects the attempt (step x 0.2) and does not fail the trajectory.
 *                State: k + 7S + R + nnz(LU) doubles per thread (nnz(LU) = nonzeros of the factor, diagonal included), 32
 *                threads at least, else VS_ERR_UNSUPPORTED.  Two-phase route only; VS_FLAG_SEPARABLE is
 *                VS_ERR_UNSUPPORTED.  Frozen arithmetic in device.cuh: MassActionStiff.
 *
 * Every objective has l outputs per point: 1 for the first three, L for MASS_ACTION, L*NT for MASS_ACTION_ADAPTIVE and
 * MASS_ACTION_STIFF (vs_objective_outputs).  The entry
 * points that take an objective write l columns: vs_eval_values rows*(2+2k)*l doubles, vs_fused_partials
 * vs_partials_len(k, l) doubles, vs_run_fused / vs_run_fused_p2p vs_result arrays sized for l. */
enum vs_objective { VS_OBJ_GFUNCTION = 0, VS_OBJ_ISHIGAMI = 1, VS_OBJ_RK4_CHAIN = 2, VS_OBJ_MASS_ACTION = 3,
                   VS_OBJ_MASS_ACTION_ADAPTIVE = 4, VS_OBJ_MASS_ACTION_STIFF = 5 };

/* fp64 arithmetic of the Halton radical inverse (the reference delegates it to the third-party ghalton package,
 * varsens/saltelli.py:82-84, whose source is not part of the reference; see DESIGN.md "parity unpinned").  The first three are
 * in-order sums of per-digit terms, least significant digit first, and differ only in how a term is rounded:
 *   DIVIDE               term = digit / b^(j+1)                       (default: ghalton as restated in oracle/halton.py)
 *   RECIPROCAL           term = digit * (1.0 / b^(j+1))
 *   RUNNING_RECIPROCAL   term = digit * f_j,  f_0 = 1.0 / b,  f_{j+1} = f_j * (1.0 / b)
 *   HORNER               x = (x + digit_j) / b from the most significant digit down (no term table: the fused kernels do not
 *                        run in this mode, the generators / export / two-phase paths do)
 * Selected per context: VS_HALTON_MODE in the environment at vs_ctx_create, or vs_ctx_set_halton_mode. */
enum vs_halton_mode { VS_HALTON_DIVIDE = 0, VS_HALTON_RECIPROCAL = 1, VS_HALTON_RUNNING_RECIPROCAL = 2, VS_HALTON_HORNER = 3 };

enum vs_flags {
    VS_FLAG_SECOND_ORDER = 1, /* also accumulate the k x k Grams for sens_2 / sens_2n */
    VS_FLAG_SEPARABLE = 2     /* product-form objectives only: evaluate the 2+2k points of a row from
                                 prefix/suffix products (O(k) instead of O(k^2)); reported separately,
                                 never used for the roofline figure */
};

/* Results of varsens/saltelli.py:572-622, host arrays the caller allocates (row-major):
 * E_2[l], var_y[l], U_j[k][l], U_nj[k][l], sens[k][l], sens_t[k][l], sens_2[k][l][k][l],
 * sens_2n[k][l][k][l].  sens_2 / sens_2n may be NULL when second order was not requested. */
typedef struct vs_result {
    double *E_2, *var_y, *U_j, *U_nj, *sens, *sens_t, *sens_2, *sens_2n;
} vs_result;

/* ---- library / context ------------------------------------------------------------------ */
int vs_abi_version(void);
const char *vs_last_error(void);
int vs_ctx_create(int device, vs_ctx **out);
int vs_ctx_destroy(vs_ctx *ctx);
/* Run on a caller stream (cudaStream_t, e.g. torch.cuda.current_stream().cuda_stream); NULL = own stream. */
int vs_ctx_set_stream(vs_ctx *ctx, void *cuda_stream);
int vs_ctx_synchronize(vs_ctx *ctx);
/* Tuning / diagnostic switches (VS_FUSED_VARIANT, VS_NO_PIPELINE, VS_GRAM_*, VS_P2P_TIMEOUT_MS, VS_HALTON_MODE, VS_TRACE ...) are
 * read from the environment once, at vs_ctx_create -- never on a launch path.  This re-reads them. */
int vs_ctx_reload_env(vs_ctx *ctx);
/* Halton arithmetic of this context (enum vs_halton_mode); drops the cached term table. */
int vs_ctx_set_halton_mode(vs_ctx *ctx, int mode);
/* Kernels launched by this ctx since creation (bench.py's gpu_launches). */
uint64_t vs_ctx_launch_count(const vs_ctx *ctx);

/* ---- host-only helpers (no GPU needed) ----------------------------------------------------- */
/* ghalton's bases: the first k primes (call site varsens/saltelli.py:82). */
int vs_halton_bases(int k, uint32_t *bases);
/* The per-digit term table the kernels sum in order: terms[offsets[d] + j*bases[d] + digit] =
 * digit / bases[d]^(j+1), j < ndigits[d] = #digits of max_index in base d.  Pass terms == NULL to
 * query *count.  This single function fixes the generator's fp64 arithmetic (swap it to re-point
 * the kernels at a different ghalton build). */
int vs_halton_terms(int k, uint64_t max_index, uint32_t *ndigits, uint32_t *offsets, double *terms,
                    uint64_t capacity, uint64_t *count);
/* The same table in any of the three term-table modes (enum vs_halton_mode); VS_HALTON_HORNER has no table: VS_ERR_UNSUPPORTED. */
int vs_halton_terms_mode(int k, uint64_t max_index, int mode, uint32_t *ndigits, uint32_t *offsets, double *terms,
                         uint64_t capacity, uint64_t *count);
/* Host-only self check of the fused kernels' computed-term form (terms of bases >= 37 are computed as the product of
 * 8*digit with a double-double reciprocal instead of being looked up): 1 if it reproduces EVERY entry of the term table of
 * `mode` bit for bit -- all digits of all positions a 32-bit index can reach, for the first k bases --, 0 if not, -1 on bad
 * arguments.  The fused kernels refuse to run when it is 0. */
int vs_halton_arith_check(int k, int mode);
/* The row order ``numpy.random.seed(seed); numpy.random.shuffle(M_2)`` produces (varsens/saltelli.py:100-101, seed = 1):
 * perm[i] = row of the unshuffled M_2 that ends up in row i.  numpy's legacy generator (MT19937, init_genrand seeding,
 * masked-rejection rk_interval) re-implemented on uint32 with look-ahead prefetching; bit-identical to numpy for every n
 * (tests/test_cabi_host.py).  key_out[624] / pos_out (optional) receive the generator state after the shuffle, so the caller
 * can leave numpy's global RNG where the reference would (numpy.random.set_state(('MT19937', key, pos, 0, 0.0))). */
int vs_reference_permutation(uint64_t n, uint32_t seed, uint32_t *perm, uint32_t *key_out, int *pos_out);
/* Length of the partial-sum vector for k factors and l outputs: 4l + m(m+1)/2, m = (2+2k) l.
 * Layout: S_A[l], S_B[l], Q_A[l], Q_B[l] (sums / sums of squares of fM_1 - c, fM_2 - c for a
 * common shift c), then the upper triangle (row-major, t <= u) of G[t][u] = sum_i v_i[t] v_i[u]
 * with v_i = (fM_1[i], fM_2[i], fN_j[0..k)[i], fN_nj[0..k)[i]) x outputs, index t*l + o.
 * vs_fused_partials may deliver the second-order blocks SYMMETRISED (J_j = fN_j[j], N_j = fN_nj[j]):
 *   G[J_i][J_j] = G[N_i][N_j] = (N_i.N_j + J_i.J_j)/2  and  G[J_i][N_j] = (N_i.J_j + J_i.N_j)/2,
 * i.e. exactly the combinations vs_finalize adds up (saltelli.py:612-613, 618-619); vectors from
 * vs_partials_from_values hold the plain entries.  Both kinds add up across shards and ranks. */
size_t vs_partials_len(int k, int l);
/* Outputs per point l of a registered objective (1, L for VS_OBJ_MASS_ACTION, L*NT for VS_OBJ_MASS_ACTION_ADAPTIVE and
 * VS_OBJ_MASS_ACTION_STIFF) in *l, after the same validation of k, objective and params the evaluating entry points run (VS_ERR_ARG on a malformed
 * description). */
int vs_objective_outputs(int k, int objective, const double *params, int n_params, int *l);

/* ---- generators ---------------------------------------------------------------------------- */
/* ghalton.Halton(k).get() points of 1-based indices first_index .. first_index+count-1, scaled;
 * out is row-major (count, k).  Replaces varsens/saltelli.py:82-84 (+ :92,95 scaling). */
int vs_halton(vs_ctx *ctx, int k, uint64_t first_index, uint64_t count, const vs_scale *scale,
              double *out, int out_mem);
/* 32-bit Gray-code Sobol points first_point .. first_point+count-1 (point 0 = origin) by direct
 * indexing; dirnums is host uint32 [k][32], MSB-aligned.  quantize6 != 0 reproduces the 6
 * significant decimal digits sobolGen prints.  Replaces quantlib/sobolGen.cpp:47-63
 * (row r of its output is point 4097 + r). */
int vs_sobol(vs_ctx *ctx, int k, uint64_t first_point, uint64_t count, const uint32_t *dirnums,
             int quantize6, const vs_scale *scale, double *out, int out_mem);

/* ---- sample assembly (export mode) ----------------------------------------------------------- */
/* Rows [row_begin,row_end) of Sample.flat() -- M_1 | M_2 | N_j[0..k) | N_nj[0..k), each n rows --
 * written row-major (row_end-row_begin, k).  perm = the row permutation of M_2 (n uint32).
 * raw == NULL: Halton source with s = 20k + discard points skipped.  raw != NULL: an unscaled
 * (2n,k) sample (Sample(raw=...) / loadFile=..., e.g. Sobol).  Replaces varsens/saltelli.py:86-125
 * (scale, shuffle, generate_N_j) and :127-160 (flat). */
int vs_sample_flat(vs_ctx *ctx, int k, uint64_t n, uint64_t discard, const uint32_t *perm, int perm_mem,
                   const double *raw, int raw_mem, const vs_scale *scale, uint64_t row_begin,
                   uint64_t row_end, double *out, int out_mem);

/* The BASE-ROW shard [i_begin,i_end) of every block of Sample.flat(): out[(t*rows + (i - i_begin))*k + c], t in [0, 2+2k),
 * rows = i_end - i_begin -- i.e. the flat layout of the sub-design made of those base rows.  This is the multi-GPU split of
 * export mode: rank r takes a contiguous range of base rows and generates only THOSE Halton points (a flat-row window of the
 * same size needs the points of nearly all n base rows).  No collective.  Replaces varsens/saltelli.py:86-160, :184-193. */
int vs_sample_flat_shard(vs_ctx *ctx, int k, uint64_t n, uint64_t discard, const uint32_t *perm, int perm_mem,
                         const double *raw, int raw_mem, const vs_scale *scale, uint64_t i_begin, uint64_t i_end,
                         double *out, int out_mem);

/* ---- objective evaluation --------------------------------------------------------------------- */
/* Objective values of base rows [i_begin,i_end) for a registered functor, sample rows generated on
 * the fly (never stored): fvals[(t*rows + (i-i_begin))*l + o], t in [0,2+2k), o in [0,l), rows = i_end-i_begin --
 * for the full range this is Objective.flat().  Replaces varsens/saltelli.py:308-353. */
int vs_eval_values(vs_ctx *ctx, int k, uint64_t n, uint64_t discard, const uint32_t *perm, int perm_mem,
                   const double *raw, int raw_mem, const vs_scale *scale, int objective,
                   const double *params, int n_params, uint64_t i_begin, uint64_t i_end, double *fvals,
                   int fvals_mem);

/* ---- estimators --------------------------------------------------------------------------------- */
/* Partial sums (vs_partials_len doubles) of `rows` base rows of objective values laid out
 * fvals[(t*rows + r)*l + o].  shift = host l doubles (common shift c, must be identical on every
 * rank; NULL = 0).  Replaces the reductions of varsens/saltelli.py:577-622. */
int vs_partials_from_values(vs_ctx *ctx, int k, int l, uint64_t rows, const double *fvals, int fvals_mem,
                            const double *shift, int flags, double *partials, int partials_mem);
/* Indices from (all-reduced) partial sums.  n = the reference's divisor (saltelli.py:577,591-596); rows =
 * base rows that actually contributed (== n unless NaN rows were trimmed, saltelli.py:474-495: var_y is the
 * unbiased variance of the 2*rows surviving values while E_2 and U keep dividing by n and n-1). */
int vs_finalize(vs_ctx *ctx, int k, int l, uint64_t n, uint64_t rows, const double *partials, int partials_mem,
                int flags, vs_result *result);
/* vs_finalize without the device-to-host copy: the 2l + 4kl + 2(kl)^2 result doubles (E_2, var_y, U_j, U_nj, sens, sens_t,
 * sens_2, sens_2n, in that order) are left in the caller's device buffer and nothing is synchronised -- the form to
 * capture in a CUDA graph together with vs_fused_partials (device buffers) and the all-reduce. */
int vs_finalize_device(vs_ctx *ctx, int k, int l, uint64_t n, uint64_t rows, const double *partials_dev, int flags,
                       double *result_dev);
/* Multi-GPU: vs_finalize fused with the all-reduce, over NVLink peer memory (no NCCL call).  ONE single-CTA kernel per
 * rank, low-latency protocol: every double of this rank's partial sums is stored as one 16-byte unit {lo, epoch, hi, epoch}
 * into slot `rank` of every peer's exchange buffer (peer_bufs[r], device pointers mapped into this process, e.g. torch
 * symmetric memory; one warp per peer); each rank then polls the tags of its own buffer -- at most VS_P2P_TIMEOUT_MS, then
 * VS_ERR_TIMEOUT --, sums the world_size slots in rank order (identical bits on every rank) and computes the indices.  No
 * fence, no separate flag.  Each peer buffer holds 2 (epoch parity) * world_size * vs_partials_len(k,l) * 16 bytes,
 * zero-initialised; epoch must start at 1 and increase by one per call on every rank.  peer_flags is ignored (kept in the
 * signature for ABI stability; may be NULL).  Replaces the file-batch gather of varsens/saltelli.py:415-472 + :572-622. */
int vs_allreduce_finalize_p2p(vs_ctx *ctx, int k, int l, uint64_t n, uint64_t rows, int world_size, int rank,
                              const uint64_t *peer_bufs, const uint64_t *peer_flags, uint32_t epoch,
                              const double *partials_dev, int flags, vs_result *result);
/* vs_partials_from_values + vs_finalize over a whole design (Objective(objective_vals=...) route,
 * varsens/saltelli.py:297-298 -> :572-622).  rows may be < n after NaN trimming (:474-495). */
int vs_indices_from_values(vs_ctx *ctx, int k, int l, uint64_t n, uint64_t rows, const double *fvals,
                           int fvals_mem, int flags, vs_result *result);

/* ---- fused pipeline ------------------------------------------------------------------------------ */
/* Generation + scaling + assembly + objective + reductions for base rows [i_begin,i_end) in one
 * kernel; sample matrices never touch HBM.  Produces this shard's partial sums; sum them over
 * ranks (one all-reduce) and call vs_finalize.  Replaces varsens/saltelli.py:82-125, :308-353 and
 * the reductions of :577-622. */
int vs_fused_partials(vs_ctx *ctx, int k, uint64_t n, uint64_t discard, const uint32_t *perm, int perm_mem,
                      const double *raw, int raw_mem, const vs_scale *scale, int objective,
                      const double *params, int n_params, uint64_t i_begin, uint64_t i_end, int flags,
                      double *partials, int partials_mem);
/* Single-GPU convenience: vs_fused_partials over [0,n) + vs_finalize.  This is
 * Varsens(objective, scaling, k, n) (varsens/saltelli.py:545-570) for a registered functor. */
int vs_run_fused(vs_ctx *ctx, int k, uint64_t n, uint64_t discard, const uint32_t *perm, int perm_mem,
                 const double *raw, int raw_mem, const vs_scale *scale, int objective, const double *params,
                 int n_params, int flags, vs_result *result);

/* Multi-GPU form of vs_run_fused: ONE kernel launch per rank and step.  Rank `rank` of `world_size` evaluates base rows
 * [i_begin,i_end) of the n-row design; the last CTA of its kernel combines the CTA sums in fixed order, stores the packed
 * partial sums into slot `rank` of every peer's exchange buffer over NVLink (one warp per peer, 16-byte {lo, epoch, hi, epoch}
 * units), polls -- at most VS_P2P_TIMEOUT_MS (default 10 s), then VS_ERR_TIMEOUT -- the tags of its own buffer, sums the slots
 * in rank order (identical bits on every rank), computes the estimators and writes them to mapped host memory.  Buffers and
 * epoch are those of vs_allreduce_finalize_p2p.  There is no NCCL call and no separate reduction, finalisation or copy
 * launch.  Replaces varsens/saltelli.py:82-125, :308-353, :572-622 and the file-batch gather of :415-472. */
int vs_run_fused_p2p(vs_ctx *ctx, int k, uint64_t n, uint64_t discard, const uint32_t *perm, int perm_mem,
                     const double *raw, int raw_mem, const vs_scale *scale, int objective, const double *params,
                     int n_params, uint64_t i_begin, uint64_t i_end, int flags, int world_size, int rank,
                     const uint64_t *peer_bufs, const uint64_t *peer_flags, uint32_t epoch, vs_result *result);

/* ---- measurement helpers --------------------------------------------------------------------------- */
/* DFMA-chain microbenchmark: returns measured FP64 TFLOP/s (FMA = 2 flops) of this GPU in *tflops. */
int vs_measure_fp64_peak(vs_ctx *ctx, double *tflops);
/* Device time in ms of the last vs_fused_partials / vs_run_fused / vs_eval_values / vs_partials_from_values /
 * vs_sample_flat main kernel, from CUDA events recorded on the ctx stream around the launch.  The events are only recorded
 * while timing is switched on (off by default: two event records are ~4 us of host time per call). */
int vs_ctx_set_timing(vs_ctx *ctx, int on);
int vs_last_kernel_ms(vs_ctx *ctx, float *ms);
/* Time stamps (ns, %globaltimer) of the tail of the last one-launch fused step with estimators (vs_run_fused /
 * vs_run_fused_p2p, k factors), taken in the CTA that finished last: {combine + pack (total), peer stores, wait for the
 * peers' elements + rank-order sum, estimators + result stores; then the parts of the first: first-level combine,
 * group row + fence + ticket, second-level combine, packing; then that CTA's own prologue, main loop and CTA-level combine}
 * -- 11 doubles. */
int vs_last_tail_ns(vs_ctx *ctx, int k, double *ns11);
/* Step counts of the last call on this ctx that evaluated a VS_OBJ_MASS_ACTION_ADAPTIVE or VS_OBJ_MASS_ACTION_STIFF network
 * (vs_eval_values,
 * vs_fused_partials, vs_run_fused, vs_run_fused_p2p), over the trajectories of its base rows [i_begin, i_end) -- not the
 * extra evaluation of base row 0 for the common shift: stats[0] accepted steps, [1] rejected steps, [2] failed trajectories,
 * [3] lane work = the sum over warps (32 consecutive rows of one design point) of rows in the warp x the most attempts of
 * any lane in it.  (accepted + rejected) / lane work is the share of lanes that did useful work.  Synchronises the ctx
 * stream; VS_ERR_ARG if no adaptive or stiff network has been evaluated on this ctx. */
int vs_last_network_stats(vs_ctx *ctx, uint64_t stats[4]);

#ifdef __cplusplus
}
#endif
#endif /* VARSENS_B200_H */
