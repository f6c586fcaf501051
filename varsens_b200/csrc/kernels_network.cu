// Mass-action reaction networks (VS_OBJ_MASS_ACTION): host validation of the packed description, and the two-phase
// evaluation kernel that integrates one trajectory per design point.  Frozen arithmetic: device.cuh, MassAction.
#include "device.cuh"

#include <cmath>
#include <vector>

namespace vs {

namespace {

constexpr int NET_MAX_S = 128, NET_MAX_R = 512, NET_MAX_L = 64;
constexpr int NET_IRREV = -2;       // kr coordinate of an irreversible reaction in the derived table
constexpr int NET_HDR = 5, NET_REC = 8;

bool int_in(double v, double lo, double hi, int *out) {
    if (!std::isfinite(v) || v != std::floor(v) || v < lo || v > hi) return false;
    *out = (int)v;
    return true;
}

}  // namespace

// Layout of the derived tables get_objective appends to the packed parameters (np doubles):
//   [np] nnz  [np+1] nobs
//   rx   R x 8:    a0 a1 b0 b1 kf_coord kf_const kr_coord kr_const   (one-species sides in slot 0; kr_coord = NET_IRREV for an
//                                                                      irreversible reaction)
//   ptr  S+1, ent nnz:   species-major stoichiometry, ent = r*8 + (c+2), c in {-2,-1,1,2}, reactions ascending per species
//   optr L+1, oent 2*nobs: observable-major (species, weight) of the nonzero weights, species ascending
struct NetLayout {
    int S, R, L, nsteps, nnz, nobs;
    double dt;
    int o_init, o_rx, o_ptr, o_ent, o_optr, o_oent;
};

static NetLayout net_layout(const double *h) {
    NetLayout n;
    n.S = (int)h[0];
    n.R = (int)h[1];
    n.L = (int)h[2];
    n.dt = h[3];
    n.nsteps = (int)h[4];
    n.o_init = NET_HDR + NET_REC * n.R;
    const int np = n.o_init + 2 * n.S + n.L * n.S;
    n.nnz = (int)h[np];
    n.nobs = (int)h[np + 1];
    n.o_rx = np + 2;
    n.o_ptr = n.o_rx + NET_REC * n.R;
    n.o_ent = n.o_ptr + n.S + 1;
    n.o_optr = n.o_ent + n.nnz;
    n.o_oent = n.o_optr + n.L + 1;
    return n;
}

int network_describe(int k, const double *p, int n_params, std::vector<double> *h, int *l) {
    VS_REQUIRE(p && n_params >= NET_HDR, VS_ERR_ARG, "mass-action network: %d parameters, the header alone has %d", n_params,
               NET_HDR);
    int S = 0, R = 0, L = 0, nsteps = 0, v = 0;
    VS_REQUIRE(int_in(p[0], 1, NET_MAX_S, &S), VS_ERR_ARG, "mass-action network: S = %g, need an integer in [1,%d]", p[0], NET_MAX_S);
    VS_REQUIRE(int_in(p[1], 1, NET_MAX_R, &R), VS_ERR_ARG, "mass-action network: R = %g, need an integer in [1,%d]", p[1], NET_MAX_R);
    VS_REQUIRE(int_in(p[2], 1, NET_MAX_L, &L), VS_ERR_ARG, "mass-action network: L = %g, need an integer in [1,%d]", p[2], NET_MAX_L);
    VS_REQUIRE(std::isfinite(p[3]), VS_ERR_ARG, "mass-action network: dt = %g is not finite", p[3]);
    VS_REQUIRE(int_in(p[4], 0, 2147483647.0, &nsteps), VS_ERR_ARG, "mass-action network: nsteps = %g, need an integer in [0,2^31)",
               p[4]);
    const long long want = NET_HDR + (long long)NET_REC * R + 2ll * S + (long long)L * S;
    VS_REQUIRE(n_params == want, VS_ERR_ARG, "mass-action network with S=%d, R=%d, L=%d needs %lld parameters, got %d", S, R, L,
               want, n_params);
    std::vector<double> rx((size_t)NET_REC * R);
    std::vector<std::vector<int>> lists(S);
    for (int r = 0; r < R; ++r) {
        const double *q = p + NET_HDR + (size_t)NET_REC * r;
        int sp[4];
        for (int e = 0; e < 4; ++e)
            VS_REQUIRE(int_in(q[e], -1, S - 1, &sp[e]), VS_ERR_ARG,
                       "mass-action network: reaction %d, species field %d = %g, need -1 or an integer in [0,%d)", r, e, q[e], S);
        int kfc = 0, krc = 0;
        VS_REQUIRE(int_in(q[4], -1, k - 1, &kfc), VS_ERR_ARG,
                   "mass-action network: reaction %d, kf coordinate %g, need -1 or an integer in [0,k=%d)", r, q[4], k);
        VS_REQUIRE(int_in(q[6], -1, k - 1, &krc), VS_ERR_ARG,
                   "mass-action network: reaction %d, kr coordinate %g, need -1 or an integer in [0,k=%d)", r, q[6], k);
        for (int side = 0; side < 2; ++side)                       // a one-species side keeps its species in slot 0
            if (sp[2 * side] < 0 && sp[2 * side + 1] >= 0) { sp[2 * side] = sp[2 * side + 1]; sp[2 * side + 1] = -1; }
        double *o = rx.data() + (size_t)NET_REC * r;
        for (int e = 0; e < 4; ++e) o[e] = sp[e];
        o[4] = kfc;
        o[5] = q[5];
        o[6] = (krc < 0 && q[7] == 0.0) ? NET_IRREV : krc;
        o[7] = q[7];
        // net stoichiometric coefficient of every species the reaction touches (a catalyst nets to 0 and is dropped)
        for (int e = 0; e < 4; ++e) {
            const int s = sp[e];
            bool first = s >= 0;
            for (int f = 0; f < e && first; ++f) first = sp[f] != s;
            if (!first) continue;
            const int c = (sp[2] == s) + (sp[3] == s) - (sp[0] == s) - (sp[1] == s);
            if (c != 0) lists[s].push_back(r * 8 + (c + 2));
        }
    }
    for (int s = 0; s < S; ++s) {
        const double *q = p + NET_HDR + (size_t)NET_REC * R + 2 * (size_t)s;
        VS_REQUIRE(int_in(q[0], -1, k - 1, &v), VS_ERR_ARG,
                   "mass-action network: species %d, initial-amount coordinate %g, need -1 or an integer in [0,k=%d)", s, q[0], k);
    }
    if (h) {
        const double *w = p + NET_HDR + (size_t)NET_REC * R + 2 * (size_t)S;
        h->assign(p, p + n_params);
        int nnz = 0, nobs = 0;
        for (int s = 0; s < S; ++s) nnz += (int)lists[s].size();
        for (int e = 0; e < L * S; ++e) nobs += w[e] != 0.0;
        h->push_back(nnz);
        h->push_back(nobs);
        h->insert(h->end(), rx.begin(), rx.end());
        int at = 0;
        for (int s = 0; s < S; ++s) { h->push_back(at); at += (int)lists[s].size(); }
        h->push_back(at);
        for (int s = 0; s < S; ++s) h->insert(h->end(), lists[s].begin(), lists[s].end());
        at = 0;
        for (int o = 0; o < L; ++o) {
            h->push_back(at);
            for (int s = 0; s < S; ++s) at += w[(size_t)o * S + s] != 0.0;
        }
        h->push_back(at);
        for (int o = 0; o < L; ++o)
            for (int s = 0; s < S; ++s)
                if (w[(size_t)o * S + s] != 0.0) { h->push_back(s); h->push_back(w[(size_t)o * S + s]); }
    }
    *l = L;
    return VS_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// One thread per design point of a base row (the work split of eval_values_kernel's heavy route: grid.y = the 2+2k points).
// The network tables live in shared memory once per CTA; every index into them is warp-uniform, so each read is a
// broadcast.  The per-trajectory state lives in shared memory too, laid out [variable][thread] (conflict-free):
//   x[k]   the point's scaled coordinates (rates and initial amounts that are coordinates read them)
//   X[S]   the state, T[S] the next stage's input, A[S] the RK4 accumulator, F[R] the fluxes of the current stage.
// A stage stores the R fluxes, then sweeps the species-major stoichiometry list: each d_s is formed in a register and folded
// into A and T (or X) at once, so no derivative array is stored.  Nothing touches global memory inside the time loop.
// ---------------------------------------------------------------------------------------------------------------------
struct NetDev {
    const double *tab;
    NetLayout n;
};

constexpr int NET_THREADS = 64;

__host__ __device__ static size_t net_table_bytes(const NetLayout &n) {
    const size_t b = 40 * (size_t)n.R + 4 * (size_t)(n.S + 1 + n.nnz);
    return (b + 15) / 16 * 16;
}

static size_t net_smem(const NetLayout &n, int k, int nthr) {
    return net_table_bytes(n) + (size_t)(k + 3 * n.S + n.R) * nthr * sizeof(double);
}

__global__ void __launch_bounds__(NET_THREADS) network_values_kernel(int k, SourceDev src, ScaleDev s, NetDev net, uint64_t i_begin,
                                                                     uint64_t i_end, double *__restrict__ fvals) {
    extern __shared__ __align__(16) double smem[];
    const NetLayout &n = net.n;
    const int S = n.S, R = n.R, nthr = blockDim.x, tid = threadIdx.x;
    double2 *rk = reinterpret_cast<double2 *>(smem);              // R: kf const, kr const
    int4 *ri = reinterpret_cast<int4 *>(rk + R);                  // R: a0 a1 b0 b1
    int2 *rc = reinterpret_cast<int2 *>(ri + R);                  // R: kf coord, kr coord
    int *cptr = reinterpret_cast<int *>(rc + R);                  // S+1
    int *cent = cptr + S + 1;                                     // nnz
    for (int r = tid; r < R; r += nthr) {
        const double *q = net.tab + n.o_rx + (size_t)NET_REC * r;
        ri[r] = make_int4((int)q[0], (int)q[1], (int)q[2], (int)q[3]);
        rc[r] = make_int2((int)q[4], (int)q[6]);
        rk[r] = make_double2(q[5], q[7]);
    }
    for (int e = tid; e <= S; e += nthr) cptr[e] = (int)net.tab[n.o_ptr + e];
    for (int e = tid; e < n.nnz; e += nthr) cent[e] = (int)net.tab[n.o_ent + e];
    __syncthreads();
    const uint64_t rows = i_end - i_begin;
    const uint64_t row = (uint64_t)blockIdx.x * nthr + tid;
    if (row >= rows) return;
    double *x = smem + net_table_bytes(n) / sizeof(double) + tid;   // x[c * nthr]
    double *X = x + (size_t)k * nthr, *T = X + (size_t)S * nthr, *A = T + (size_t)S * nthr, *F = A + (size_t)S * nthr;
    const uint64_t i = i_begin + row, pi = src.perm[i];
    const int p = blockIdx.y;
    const int j = p < 2 ? -1 : (p < 2 + k ? p - 2 : p - 2 - k);
    const bool base_a = p == 0 || p >= 2 + k;                     // M_1 and N_nj start from A_i, M_2 and N_j from B_i
    for (int c = 0; c < k; ++c) {
        const bool from_a = (c == j) ? !base_a : base_a;
        x[c * nthr] = from_a ? apply_scale(s, c, source_a(src, k, i, c)) : apply_scale(s, c, source_b(src, k, pi, c));
    }
    for (int sp = 0; sp < S; ++sp) {
        const double *q = net.tab + n.o_init + 2 * sp;
        const int ic = (int)q[0];
        X[sp * nthr] = ic >= 0 ? x[ic * nthr] : q[1];
    }
    const double dt = n.dt, h2 = __dmul_rn(0.5, dt), h6 = __ddiv_rn(dt, 6.0);
    // fluxes of state Y into F
    auto fluxes = [&](const double *Y) {
#pragma unroll 4
        for (int r = 0; r < R; ++r) {
            const int4 sp = ri[r];
            const int2 cc = rc[r];
            const double2 kc = rk[r];
            const double kf = cc.x >= 0 ? x[cc.x * nthr] : kc.x;
            const double pf = sp.x < 0 ? 1.0 : (sp.y < 0 ? Y[sp.x * nthr] : __dmul_rn(Y[sp.x * nthr], Y[sp.y * nthr]));
            double f;
            if (cc.y == NET_IRREV) {
                f = __dmul_rn(kf, pf);
            } else {
                const double kr = cc.y >= 0 ? x[cc.y * nthr] : kc.y;
                const double pr = sp.z < 0 ? 1.0 : (sp.w < 0 ? Y[sp.z * nthr] : __dmul_rn(Y[sp.z * nthr], Y[sp.w * nthr]));
                f = fma(kf, pf, -__dmul_rn(kr, pr));
            }
            F[r * nthr] = f;
        }
    };
    // d_s of species sp from the stored fluxes, ascending reaction order
    auto deriv = [&](int sp) {
        double d = 0.0;
        const int e1 = cptr[sp + 1];
        for (int e = cptr[sp]; e < e1; ++e) {
            const int code = cent[e];
            const int c = (code & 7) - 2;
            const double fl = F[(code >> 3) * nthr];
            if (c == 1) d = __dadd_rn(d, fl);
            else if (c == -1) d = __dsub_rn(d, fl);
            else d = fma((double)c, fl, d);
        }
        return d;
    };
    for (int it = 0; it < n.nsteps; ++it) {
        fluxes(X);                                                // k1
        for (int sp = 0; sp < S; ++sp) {
            const double d = deriv(sp);
            A[sp * nthr] = d;
            T[sp * nthr] = fma(h2, d, X[sp * nthr]);
        }
        fluxes(T);                                                // k2
        for (int sp = 0; sp < S; ++sp) {
            const double d = deriv(sp);
            A[sp * nthr] = fma(2.0, d, A[sp * nthr]);
            T[sp * nthr] = fma(h2, d, X[sp * nthr]);
        }
        fluxes(T);                                                // k3
        for (int sp = 0; sp < S; ++sp) {
            const double d = deriv(sp);
            A[sp * nthr] = fma(2.0, d, A[sp * nthr]);
            T[sp * nthr] = fma(dt, d, X[sp * nthr]);
        }
        fluxes(T);                                                // k4
        for (int sp = 0; sp < S; ++sp) {
            const double d = deriv(sp);
            X[sp * nthr] = fma(h6, __dadd_rn(A[sp * nthr], d), X[sp * nthr]);
        }
    }
    const int L = n.L;
    double *out = fvals + ((uint64_t)p * rows + row) * L;
    for (int o = 0; o < L; ++o) {
        double acc = 0.0;
        const int e1 = (int)net.tab[n.o_optr + o + 1];
        for (int e = (int)net.tab[n.o_optr + o]; e < e1; ++e) {
            const double *q = net.tab + n.o_oent + 2 * e;
            acc = fma(q[1], X[(int)q[0] * nthr], acc);
        }
        out[o] = acc;
    }
}

int network_check_fit(vs_ctx *c, int k, const ObjectiveDev &o) {
    const NetLayout n = net_layout(o.host);
    VS_REQUIRE(net_smem(n, k, 32) <= c->smem_optin, VS_ERR_UNSUPPORTED,
               "mass-action network with k=%d, S=%d, R=%d needs %zu bytes of shared memory for 32 trajectories, the device has %zu",
               k, n.S, n.R, net_smem(n, k, 32), c->smem_optin);
    return VS_OK;
}

int launch_network_values(vs_ctx *c, int k, const SourceDev &src, const ScaleDev &s, const ObjectiveDev &o, uint64_t i_begin,
                          uint64_t i_end, double *fvals) {
    VS_TRY(network_check_fit(c, k, o));
    const uint64_t rows = i_end - i_begin;
    if (rows == 0) return VS_OK;
    NetDev net{o.params, net_layout(o.host)};
    const int nthr = net_smem(net.n, k, NET_THREADS) <= c->smem_optin ? NET_THREADS : 32;
    const size_t smem = net_smem(net.n, k, nthr);
    VS_CUDA(cudaFuncSetAttribute(network_values_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((unsigned)((rows + nthr - 1) / nthr), (unsigned)(2 + 2 * k));
    time_begin(c);
    network_values_kernel<<<grid, nthr, smem, c->stream>>>(k, src, s, net, i_begin, i_end, fvals);
    time_end(c);
    c->launches++;
    VS_CUDA(cudaGetLastError());
    if (!c->opt.trace.empty()) {                      // VS_TRACE: the form that ran (64 or 32 trajectories per CTA) and its grid
        if (FILE *fp = fopen(c->opt.trace.c_str(), "a")) {
            fprintf(fp, "# network_values_kernel nthr=%d gx=%u gy=%u smem=%zu rows=%llu\n", nthr, grid.x, grid.y, smem,
                    (unsigned long long)rows);
            fclose(fp);
        }
    }
    return VS_OK;
}

}  // namespace vs
