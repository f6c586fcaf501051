// Mass-action reaction networks (VS_OBJ_MASS_ACTION, VS_OBJ_MASS_ACTION_ADAPTIVE, VS_OBJ_MASS_ACTION_STIFF): host validation of
// the packed description, and the two-phase evaluation kernels that integrate one trajectory per design point, by fixed-step
// RK4, by adaptive Dormand-Prince 5(4) or by adaptive Rosenbrock Rodas3.  Frozen arithmetic: device.cuh, MassAction,
// MassActionAdaptive and MassActionStiff.
#include "device.cuh"

#include <algorithm>
#include <cmath>
#include <vector>

namespace vs {

namespace {

constexpr int NET_MAX_S = 128, NET_MAX_R = 512, NET_MAX_L = 64;
constexpr int NET_IRREV = -2;       // kr coordinate of an irreversible reaction in the derived table
constexpr int NET_HDR = 5, NET_HDR_ADAPTIVE = 8, NET_REC = 8;

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
// An adaptive or stiff description (NT > 0) has its NT output times at o_times, after the weights.  A stiff description
// appends the Rosenbrock tables after oent (network_describe: stiff_program).
struct NetLayout {
    int S, R, L, nsteps, nnz, nobs;
    double dt;
    int o_init, o_rx, o_ptr, o_ent, o_optr, o_oent;
    int NT, max_steps, o_times;               // NT = 0: fixed step
    double rtol, atol, h0;
    bool stiff;
    int nlu, ncol, njt, nlow, nup, nupd;      // factor slots and list lengths of the stiff tables
    int o_stiff;                              // the first of them: jptr
};

static NetLayout net_layout(const double *h, int objective) {
    NetLayout n{};
    n.S = (int)h[0];
    n.R = (int)h[1];
    n.L = (int)h[2];
    int hdr = NET_HDR;
    if (objective == VS_OBJ_MASS_ACTION_ADAPTIVE || objective == VS_OBJ_MASS_ACTION_STIFF) {
        hdr = NET_HDR_ADAPTIVE;
        n.NT = (int)h[3];
        n.rtol = h[4];
        n.atol = h[5];
        n.h0 = h[6];
        n.max_steps = (int)h[7];
    } else {
        n.dt = h[3];
        n.nsteps = (int)h[4];
    }
    n.o_init = hdr + NET_REC * n.R;
    n.o_times = n.o_init + 2 * n.S + n.L * n.S;
    const int np = n.o_times + n.NT;
    n.nnz = (int)h[np];
    n.nobs = (int)h[np + 1];
    n.o_rx = np + 2;
    n.o_ptr = n.o_rx + NET_REC * n.R;
    n.o_ent = n.o_ptr + n.S + 1;
    n.o_optr = n.o_ent + n.nnz;
    n.o_oent = n.o_optr + n.L + 1;
    n.stiff = objective == VS_OBJ_MASS_ACTION_STIFF;
    if (n.stiff) {
        const double *c = h + n.o_oent + 2 * n.nobs;
        n.nlu = (int)c[0];
        n.ncol = (int)c[1];
        n.njt = (int)c[2];
        n.nlow = (int)c[3];
        n.nup = (int)c[4];
        n.nupd = (int)c[5];
        n.o_stiff = n.o_oent + 2 * n.nobs + 6;
    }
    return n;
}

// Rosenbrock tables of a stiff description, appended to h after the observable lists (all entries exact integers):
//   nlu ncol njt nlow nup nupd
//   jptr R+1, jcol ncol   Jacobian scatter: the columns of reaction r, jcol[jptr[r] .. jptr[r+1]), species ascending: its
//                         reactants (catalysts included), and its products if it is reversible
//   jtp ncol+1, jt njt    targets of column e, jt[jtp[e] .. jtp[e+1]) = slot*8 + (nu+2) for each species with net coefficient
//                         nu != 0 in the reaction, species ascending; slot = the factor slot of (species, column)
//   ord S, piv S          elimination order: the species at position p, and the factor slot of its pivot
//   lptr S+1, lent nlow   column p of L below the pivot, positions ascending: slot*128 + species
//   uptr S+1, uent nup    row p of U right of the pivot, positions ascending: slot*128 + species
//   upd nupd              target slots of pivot p's update: for each L entry of p in order, for each U entry of p in order
// Pattern: entry (s, c) is the diagonal, or some reaction has a nonzero net coefficient for s and c among its columns.  Order:
// minimum degree on the symmetrised pattern (repeatedly eliminate the remaining species of least degree, ties to the lowest
// index, and connect its remaining neighbours); factor pattern: symbolic LU without pivoting in that order.  Slots number the
// factor's entries row-major in elimination positions.
static void stiff_program(int S, int R, const std::vector<double> &rx, const std::vector<std::vector<int>> &lists,
                          std::vector<double> *h) {
    std::vector<std::vector<std::pair<int, int>>> nu(R);        // (species, nu) per reaction, species ascending
    for (int s = 0; s < S; ++s)
        for (int code : lists[s]) nu[code >> 3].push_back({s, (code & 7) - 2});
    std::vector<std::vector<int>> cols(R);
    std::vector<char> P((size_t)S * S, 0);                      // species pattern
    for (int s = 0; s < S; ++s) P[(size_t)s * S + s] = 1;
    for (int r = 0; r < R; ++r) {
        const double *q = rx.data() + (size_t)NET_REC * r;
        const bool rev = (int)q[6] != NET_IRREV;
        for (int e = 0; e < (rev ? 4 : 2); ++e)
            if (q[e] >= 0) cols[r].push_back((int)q[e]);
        std::sort(cols[r].begin(), cols[r].end());
        cols[r].erase(std::unique(cols[r].begin(), cols[r].end()), cols[r].end());
        for (auto sv : nu[r])
            for (int c : cols[r]) P[(size_t)sv.first * S + c] = 1;
    }
    std::vector<char> G((size_t)S * S, 0), alive(S, 1);         // elimination graph of the symmetrised pattern
    for (int a = 0; a < S; ++a)
        for (int b = 0; b < S; ++b)
            if (a != b && (P[(size_t)a * S + b] || P[(size_t)b * S + a])) G[(size_t)a * S + b] = 1;
    std::vector<int> ord(S), pos(S);
    for (int p = 0; p < S; ++p) {
        int best = -1, bd = 0;
        for (int v = 0; v < S; ++v) {
            if (!alive[v]) continue;
            int d = 0;
            for (int u = 0; u < S; ++u) d += alive[u] && G[(size_t)v * S + u];
            if (best < 0 || d < bd) { best = v; bd = d; }
        }
        alive[best] = 0;
        for (int u = 0; u < S; ++u)
            for (int w = 0; w < S; ++w)
                if (u != w && alive[u] && alive[w] && G[(size_t)best * S + u] && G[(size_t)best * S + w]) G[(size_t)u * S + w] = 1;
        ord[p] = best;
        pos[best] = p;
    }
    std::vector<char> F((size_t)S * S);                         // factor pattern in positions
    for (int i = 0; i < S; ++i)
        for (int j = 0; j < S; ++j) F[(size_t)i * S + j] = P[(size_t)ord[i] * S + ord[j]];
    for (int p = 0; p < S; ++p)
        for (int i = p + 1; i < S; ++i)
            if (F[(size_t)i * S + p])
                for (int j = p + 1; j < S; ++j)
                    if (F[(size_t)p * S + j]) F[(size_t)i * S + j] = 1;
    std::vector<int> slot((size_t)S * S, -1);
    int nlu = 0;
    for (size_t e = 0; e < F.size(); ++e)
        if (F[e]) slot[e] = nlu++;
    std::vector<int> jptr, jcol, jtp, jt, piv, lptr, lent, uptr, uent, upd;
    for (int r = 0; r < R; ++r) {
        jptr.push_back((int)jcol.size());
        for (int c : cols[r]) {
            jcol.push_back(c);
            jtp.push_back((int)jt.size());
            for (auto sv : nu[r]) jt.push_back(slot[(size_t)pos[sv.first] * S + pos[c]] * 8 + sv.second + 2);
        }
    }
    jptr.push_back((int)jcol.size());
    jtp.push_back((int)jt.size());
    for (int p = 0; p < S; ++p) {
        piv.push_back(slot[(size_t)p * S + p]);
        lptr.push_back((int)lent.size());
        uptr.push_back((int)uent.size());
        for (int i = p + 1; i < S; ++i)
            if (F[(size_t)i * S + p]) lent.push_back(slot[(size_t)i * S + p] * 128 + ord[i]);
        for (int j = p + 1; j < S; ++j)
            if (F[(size_t)p * S + j]) uent.push_back(slot[(size_t)p * S + j] * 128 + ord[j]);
        for (int i = p + 1; i < S; ++i)
            if (F[(size_t)i * S + p])
                for (int j = p + 1; j < S; ++j)
                    if (F[(size_t)p * S + j]) upd.push_back(slot[(size_t)i * S + j]);
    }
    lptr.push_back((int)lent.size());
    uptr.push_back((int)uent.size());
    for (int v : {nlu, (int)jcol.size(), (int)jt.size(), (int)lent.size(), (int)uent.size(), (int)upd.size()}) h->push_back(v);
    for (const std::vector<int> *a : {&jptr, &jcol, &jtp, &jt, &ord, &piv, &lptr, &lent, &uptr, &uent, &upd})
        h->insert(h->end(), a->begin(), a->end());
}

int network_describe(int k, int objective, const double *p, int n_params, std::vector<double> *h, int *l) {
    const bool adaptive = objective == VS_OBJ_MASS_ACTION_ADAPTIVE || objective == VS_OBJ_MASS_ACTION_STIFF;
    const int hdr = adaptive ? NET_HDR_ADAPTIVE : NET_HDR;
    VS_REQUIRE(p && n_params >= hdr, VS_ERR_ARG, "mass-action network: %d parameters, the header alone has %d", n_params, hdr);
    int S = 0, R = 0, L = 0, nsteps = 0, NT = 0, v = 0;
    VS_REQUIRE(int_in(p[0], 1, NET_MAX_S, &S), VS_ERR_ARG, "mass-action network: S = %g, need an integer in [1,%d]", p[0], NET_MAX_S);
    VS_REQUIRE(int_in(p[1], 1, NET_MAX_R, &R), VS_ERR_ARG, "mass-action network: R = %g, need an integer in [1,%d]", p[1], NET_MAX_R);
    VS_REQUIRE(int_in(p[2], 1, NET_MAX_L, &L), VS_ERR_ARG, "mass-action network: L = %g, need an integer in [1,%d]", p[2], NET_MAX_L);
    if (adaptive) {
        VS_REQUIRE(int_in(p[3], 1, NET_MAX_L, &NT) && L * NT <= NET_MAX_L, VS_ERR_ARG,
                   "adaptive mass-action network: NT = %g output times of L = %d observables, need NT >= 1 and L*NT <= %d", p[3], L,
                   NET_MAX_L);
        VS_REQUIRE(std::isfinite(p[4]) && p[4] >= 0.0, VS_ERR_ARG, "adaptive mass-action network: rtol = %g, need finite >= 0", p[4]);
        VS_REQUIRE(std::isfinite(p[5]) && p[5] > 0.0, VS_ERR_ARG, "adaptive mass-action network: atol = %g, need finite > 0", p[5]);
        VS_REQUIRE(std::isfinite(p[6]) && p[6] > 0.0, VS_ERR_ARG, "adaptive mass-action network: h0 = %g, need finite > 0", p[6]);
        VS_REQUIRE(int_in(p[7], 1, 2147483647.0, &v), VS_ERR_ARG,
                   "adaptive mass-action network: max_steps = %g, need an integer in [1,2^31)", p[7]);
    } else {
        VS_REQUIRE(std::isfinite(p[3]), VS_ERR_ARG, "mass-action network: dt = %g is not finite", p[3]);
        VS_REQUIRE(int_in(p[4], 0, 2147483647.0, &nsteps), VS_ERR_ARG,
                   "mass-action network: nsteps = %g, need an integer in [0,2^31)", p[4]);
    }
    const long long want = hdr + (long long)NET_REC * R + 2ll * S + (long long)L * S + NT;
    VS_REQUIRE(n_params == want, VS_ERR_ARG, "mass-action network with S=%d, R=%d, L=%d, NT=%d needs %lld parameters, got %d", S, R,
               L, NT, want, n_params);
    const double *times = p + want - NT;
    for (int m = 0; m < NT; ++m)
        VS_REQUIRE(std::isfinite(times[m]) && times[m] > (m ? times[m - 1] : 0.0), VS_ERR_ARG,
                   "adaptive mass-action network: output time %d = %g, need finite times with 0 < t_1 < t_2 < ...", m + 1, times[m]);
    std::vector<double> rx((size_t)NET_REC * R);
    std::vector<std::vector<int>> lists(S);
    for (int r = 0; r < R; ++r) {
        const double *q = p + hdr + (size_t)NET_REC * r;
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
        const double *q = p + hdr + (size_t)NET_REC * R + 2 * (size_t)s;
        VS_REQUIRE(int_in(q[0], -1, k - 1, &v), VS_ERR_ARG,
                   "mass-action network: species %d, initial-amount coordinate %g, need -1 or an integer in [0,k=%d)", s, q[0], k);
    }
    if (h) {
        const double *w = p + hdr + (size_t)NET_REC * R + 2 * (size_t)S;
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
        if (objective == VS_OBJ_MASS_ACTION_STIFF) stiff_program(S, R, rx, lists, h);
    }
    *l = adaptive ? L * NT : L;
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

// The reaction and stoichiometry tables in shared memory (net_load_tables).
struct NetTables {
    const double2 *rk;      // R: kf const, kr const
    const int4 *ri;         // R: a0 a1 b0 b1
    const int2 *rc;         // R: kf coord, kr coord
    const int *cptr;        // S+1
    const int *cent;        // nnz
};

constexpr int NET_THREADS = 64;

__host__ __device__ static size_t net_table_bytes(const NetLayout &n) {
    const size_t b = 40 * (size_t)n.R + 4 * (size_t)(n.S + 1 + n.nnz);
    return (b + 15) / 16 * 16;
}

// The adaptive kernel adds the output times and the observable lists (times[NT], weights[nobs], optr[L+1], species[nobs]), so
// that its step loop reads nothing from global memory.
__host__ __device__ static size_t net_adaptive_table_bytes(const NetLayout &n) {
    const size_t b = 8 * (size_t)(n.NT + n.nobs) + 4 * (size_t)(n.L + 1 + n.nobs);
    return net_table_bytes(n) + (b + 15) / 16 * 16;
}

// The Rosenbrock kernel adds the stiff tables of network_describe (jptr .. upd, one int each).
__host__ __device__ static size_t net_stiff_table_bytes(const NetLayout &n) {
    const size_t b = 4 * (size_t)(4 * n.S + n.R + 4 + 2 * n.ncol + n.njt + n.nlow + n.nup + n.nupd);
    return net_adaptive_table_bytes(n) + (b + 15) / 16 * 16;
}

static size_t net_smem(const NetLayout &n, int k, int nthr) {
    if (n.stiff) return net_stiff_table_bytes(n) + (size_t)(k + 7 * n.S + n.R + n.nlu) * nthr * sizeof(double);
    if (n.NT) return net_adaptive_table_bytes(n) + (size_t)(k + 8 * n.S + n.R) * nthr * sizeof(double);
    return net_table_bytes(n) + (size_t)(k + 3 * n.S + n.R) * nthr * sizeof(double);
}

// Every thread of the CTA copies its share of the tables; the caller synchronises.
__device__ __forceinline__ NetTables net_load_tables(double *smem, const NetDev &net) {
    const NetLayout &n = net.n;
    const int S = n.S, R = n.R, nthr = blockDim.x, tid = threadIdx.x;
    double2 *rk = reinterpret_cast<double2 *>(smem);
    int4 *ri = reinterpret_cast<int4 *>(rk + R);
    int2 *rc = reinterpret_cast<int2 *>(ri + R);
    int *cptr = reinterpret_cast<int *>(rc + R);
    int *cent = cptr + S + 1;
    for (int r = tid; r < R; r += nthr) {
        const double *q = net.tab + n.o_rx + (size_t)NET_REC * r;
        ri[r] = make_int4((int)q[0], (int)q[1], (int)q[2], (int)q[3]);
        rc[r] = make_int2((int)q[4], (int)q[6]);
        rk[r] = make_double2(q[5], q[7]);
    }
    for (int e = tid; e <= S; e += nthr) cptr[e] = (int)net.tab[n.o_ptr + e];
    for (int e = tid; e < n.nnz; e += nthr) cent[e] = (int)net.tab[n.o_ent + e];
    return NetTables{rk, ri, rc, cptr, cent};
}

// The scaled coordinates x of design point p (grid.y) of base row i, and the initial state X.
__device__ __forceinline__ void net_point(int k, const SourceDev &src, const ScaleDev &s, const NetDev &net, uint64_t i, int p,
                                          double *x, double *X, int nthr) {
    const uint64_t pi = src.perm[i];
    const int j = p < 2 ? -1 : (p < 2 + k ? p - 2 : p - 2 - k);
    const bool base_a = p == 0 || p >= 2 + k;                     // M_1 and N_nj start from A_i, M_2 and N_j from B_i
    for (int c = 0; c < k; ++c) {
        const bool from_a = (c == j) ? !base_a : base_a;
        x[c * nthr] = from_a ? apply_scale(s, c, source_a(src, k, i, c)) : apply_scale(s, c, source_b(src, k, pi, c));
    }
    for (int sp = 0; sp < net.n.S; ++sp) {
        const double *q = net.tab + net.n.o_init + 2 * sp;
        const int ic = (int)q[0];
        X[sp * nthr] = ic >= 0 ? x[ic * nthr] : q[1];
    }
}

// fluxes of state Y into F
__device__ __forceinline__ void net_fluxes(const NetTables &t, int R, int nthr, const double *x, const double *Y, double *F) {
#pragma unroll 4
    for (int r = 0; r < R; ++r) {
        const int4 sp = t.ri[r];
        const int2 cc = t.rc[r];
        const double2 kc = t.rk[r];
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
}

// d_s of species sp from the stored fluxes, ascending reaction order
__device__ __forceinline__ double net_deriv(const NetTables &t, int nthr, const double *F, int sp) {
    double d = 0.0;
    const int e1 = t.cptr[sp + 1];
    for (int e = t.cptr[sp]; e < e1; ++e) {
        const int code = t.cent[e];
        const int c = (code & 7) - 2;
        const double fl = F[(code >> 3) * nthr];
        if (c == 1) d = __dadd_rn(d, fl);
        else if (c == -1) d = __dsub_rn(d, fl);
        else d = fma((double)c, fl, d);
    }
    return d;
}

__global__ void __launch_bounds__(NET_THREADS) network_values_kernel(int k, SourceDev src, ScaleDev s, NetDev net, uint64_t i_begin,
                                                                     uint64_t i_end, double *__restrict__ fvals) {
    extern __shared__ __align__(16) double smem[];
    const NetLayout &n = net.n;
    const int S = n.S, R = n.R, nthr = blockDim.x, tid = threadIdx.x;
    const NetTables tb = net_load_tables(smem, net);
    __syncthreads();
    const uint64_t rows = i_end - i_begin;
    const uint64_t row = (uint64_t)blockIdx.x * nthr + tid;
    if (row >= rows) return;
    double *x = smem + net_table_bytes(n) / sizeof(double) + tid;   // x[c * nthr]
    double *X = x + (size_t)k * nthr, *T = X + (size_t)S * nthr, *A = T + (size_t)S * nthr, *F = A + (size_t)S * nthr;
    const int p = blockIdx.y;
    net_point(k, src, s, net, i_begin + row, p, x, X, nthr);
    const double dt = n.dt, h2 = __dmul_rn(0.5, dt), h6 = __ddiv_rn(dt, 6.0);
    for (int it = 0; it < n.nsteps; ++it) {
        net_fluxes(tb, R, nthr, x, X, F);                         // k1
        for (int sp = 0; sp < S; ++sp) {
            const double d = net_deriv(tb, nthr, F, sp);
            A[sp * nthr] = d;
            T[sp * nthr] = fma(h2, d, X[sp * nthr]);
        }
        net_fluxes(tb, R, nthr, x, T, F);                         // k2
        for (int sp = 0; sp < S; ++sp) {
            const double d = net_deriv(tb, nthr, F, sp);
            A[sp * nthr] = fma(2.0, d, A[sp * nthr]);
            T[sp * nthr] = fma(h2, d, X[sp * nthr]);
        }
        net_fluxes(tb, R, nthr, x, T, F);                         // k3
        for (int sp = 0; sp < S; ++sp) {
            const double d = net_deriv(tb, nthr, F, sp);
            A[sp * nthr] = fma(2.0, d, A[sp * nthr]);
            T[sp * nthr] = fma(dt, d, X[sp * nthr]);
        }
        net_fluxes(tb, R, nthr, x, T, F);                         // k4
        for (int sp = 0; sp < S; ++sp) {
            const double d = net_deriv(tb, nthr, F, sp);
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

// ---------------------------------------------------------------------------------------------------------------------
// Adaptive Dormand-Prince 5(4) (VS_OBJ_MASS_ACTION_ADAPTIVE): the work split and tables of network_values_kernel, plus the
// output times and observable lists in shared memory.  Per-trajectory state, [variable][thread]:
//   x[k], X[S] the state at t, Y[S] the stage input (Y7 = the 5th-order solution), K[6][S] the stage derivatives K1..K6 (K7 is
//   written into K2's slot, dead after stage 6; on acceptance the two slots swap roles, so K7 becomes the next K1: FSAL), F[R].
// Each trajectory picks its own steps; a step that would pass the next output time is clipped to land on it, and the L
// observables are written there.  Nothing else touches global memory inside the step loop.  Counts (accepted, rejected,
// failed, lane work) are reduced per warp and added with one atomicAdd each when `stats` is set.
// ---------------------------------------------------------------------------------------------------------------------
namespace dp5 {   // Hairer-Norsett-Wanner I, Table 5.2; each coefficient the correctly rounded double of its rational
constexpr double A21 = 1.0 / 5.0;
constexpr double A31 = 3.0 / 40.0, A32 = 9.0 / 40.0;
constexpr double A41 = 44.0 / 45.0, A42 = -56.0 / 15.0, A43 = 32.0 / 9.0;
constexpr double A51 = 19372.0 / 6561.0, A52 = -25360.0 / 2187.0, A53 = 64448.0 / 6561.0, A54 = -212.0 / 729.0;
constexpr double A61 = 9017.0 / 3168.0, A62 = -355.0 / 33.0, A63 = 46732.0 / 5247.0, A64 = 49.0 / 176.0, A65 = -5103.0 / 18656.0;
constexpr double A71 = 35.0 / 384.0, A73 = 500.0 / 1113.0, A74 = 125.0 / 192.0, A75 = -2187.0 / 6784.0, A76 = 11.0 / 84.0;
// e_j = b_j - bhat_j (b = row 7 of a)
constexpr double E1 = 71.0 / 57600.0, E3 = -71.0 / 16695.0, E4 = 71.0 / 1920.0, E5 = -17253.0 / 339200.0, E6 = 22.0 / 525.0,
                 E7 = -1.0 / 40.0;
}  // namespace dp5

// Y = fma(h, acc, X) with acc = fma(a_j, K_j, acc) from 0.0 over the NJ given stages, ascending
template <int NJ>
__device__ __forceinline__ void dp5_stage_input(const double (&a)[NJ], const double *const (&K)[NJ], double h, const double *X,
                                                double *Y, int S, int nthr) {
    for (int sp = 0; sp < S; ++sp) {
        double acc = 0.0;
#pragma unroll
        for (int j = 0; j < NJ; ++j) acc = fma(a[j], K[j][sp * nthr], acc);
        Y[sp * nthr] = fma(h, acc, X[sp * nthr]);
    }
}

__device__ __forceinline__ void net_rhs(const NetTables &t, int S, int R, int nthr, const double *x, const double *Y, double *F,
                                        double *D) {
    net_fluxes(t, R, nthr, x, Y, F);
    for (int sp = 0; sp < S; ++sp) D[sp * nthr] = net_deriv(t, nthr, F, sp);
}

// The output times and observable lists of the adaptive and stiff kernels in shared memory, after the network tables.
struct NetOutputs {
    const double *tout;     // NT output times
    const double *ow;       // nobs observable weights
    const int *optr;        // L+1
    const int *osp;         // nobs species
};

__device__ __forceinline__ NetOutputs net_load_outputs(double *smem, const NetDev &net) {
    const NetLayout &n = net.n;
    const int nthr = blockDim.x, tid = threadIdx.x;
    double *tout = smem + net_table_bytes(n) / sizeof(double);
    double *ow = tout + n.NT;
    int *optr = reinterpret_cast<int *>(ow + n.nobs);
    int *osp = optr + n.L + 1;
    for (int e = tid; e < n.NT; e += nthr) tout[e] = net.tab[n.o_times + e];
    for (int e = tid; e <= n.L; e += nthr) optr[e] = (int)net.tab[n.o_optr + e];
    for (int e = tid; e < n.nobs; e += nthr) {
        osp[e] = (int)net.tab[n.o_oent + 2 * e];
        ow[e] = net.tab[n.o_oent + 2 * e + 1];
    }
    return NetOutputs{tout, ow, optr, osp};
}

// The step to attempt from t towards output time `to`: h, or clipped to land on `to`.  false: the trajectory has failed
// (max_steps attempts, or a step that no longer advances t), and its outputs from output time m on are NaN.
__device__ __forceinline__ bool net_next_step(double t, double h, double to, unsigned attempts, unsigned max_steps, int m, int L,
                                              int NT, double *out, double &hs, bool &clip) {
    hs = h;
    clip = __dadd_rn(t, hs) >= to;
    if (clip) hs = __dsub_rn(to, t);
    if (attempts == max_steps || __dadd_rn(t, hs) == t) {
        for (int e = m * L; e < NT * L; ++e) out[e] = __longlong_as_double(0x7ff8000000000000ll);
        return false;
    }
    return true;
}

// The L observables of state X into out[0 .. L)
__device__ __forceinline__ void net_observe(const NetOutputs &ot, int L, int nthr, const double *X, double *out) {
    for (int o = 0; o < L; ++o) {
        double acc = 0.0;
        for (int e = ot.optr[o]; e < ot.optr[o + 1]; ++e) acc = fma(ot.ow[e], X[ot.osp[e] * nthr], acc);
        out[o] = acc;
    }
}

// vs_last_network_stats: the warp's accepted and rejected steps, failed trajectories and lane work, one atomicAdd each.
// Every lane of the warp calls it.
__device__ __forceinline__ void net_add_stats(unsigned long long *stats, bool valid, unsigned attempts, unsigned accepted,
                                              bool failed) {
    unsigned long long a = accepted, r = attempts - accepted, f = failed;
    for (int o = 16; o; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        r += __shfl_xor_sync(0xffffffffu, r, o);
        f += __shfl_xor_sync(0xffffffffu, f, o);
    }
    const unsigned most = __reduce_max_sync(0xffffffffu, attempts);
    const unsigned lanes = __popc(__ballot_sync(0xffffffffu, valid));
    if ((threadIdx.x & 31) == 0 && lanes) {
        atomicAdd(stats + 0, a);
        atomicAdd(stats + 1, r);
        atomicAdd(stats + 2, f);
        atomicAdd(stats + 3, (unsigned long long)lanes * most);
    }
}

__global__ void __launch_bounds__(NET_THREADS) network_adaptive_kernel(int k, SourceDev src, ScaleDev s, NetDev net, uint64_t i_begin,
                                                                       uint64_t i_end, double *__restrict__ fvals,
                                                                       unsigned long long *__restrict__ stats) {
    extern __shared__ __align__(16) double smem[];
    const NetLayout &n = net.n;
    const int S = n.S, R = n.R, L = n.L, NT = n.NT, nthr = blockDim.x, tid = threadIdx.x;
    const NetTables tb = net_load_tables(smem, net);
    const NetOutputs ot = net_load_outputs(smem, net);
    __syncthreads();
    const uint64_t rows = i_end - i_begin;
    const uint64_t row = (uint64_t)blockIdx.x * nthr + tid;
    const bool valid = row < rows;                                 // every lane stays for the warp reduction of the counts
    unsigned attempts = 0, accepted = 0;
    bool failed = false;
    if (valid) {
        double *x = smem + net_adaptive_table_bytes(n) / sizeof(double) + tid;
        const size_t sl = (size_t)S * nthr;
        double *X = x + (size_t)k * nthr, *Y = X + sl, *Kb = Y + sl, *F = Kb + 6 * sl;
        const int p = blockIdx.y;
        net_point(k, src, s, net, i_begin + row, p, x, X, nthr);
        double *out = fvals + ((uint64_t)p * rows + row) * (uint64_t)(L * NT);
        const double rtol = n.rtol, atol = n.atol;
        const unsigned max_steps = (unsigned)n.max_steps;
        int k1 = 0;                                                // slot of K1; K2 (and K7) in slot 1 - k1
        net_rhs(tb, S, R, nthr, x, X, F, Kb);
        double t = 0.0, h = n.h0;
        bool after_reject = false;
        for (int m = 0; m < NT;) {
            const double to = ot.tout[m];
            double hs;
            bool clip;
            if (!net_next_step(t, h, to, attempts, max_steps, m, L, NT, out, hs, clip)) {
                failed = true;
                break;
            }
            ++attempts;
            const double *K1 = Kb + k1 * sl;
            double *K2 = Kb + (1 - k1) * sl, *K3 = Kb + 2 * sl, *K4 = Kb + 3 * sl, *K5 = Kb + 4 * sl, *K6 = Kb + 5 * sl;
            dp5_stage_input<1>({dp5::A21}, {K1}, hs, X, Y, S, nthr);
            net_rhs(tb, S, R, nthr, x, Y, F, K2);
            dp5_stage_input<2>({dp5::A31, dp5::A32}, {K1, K2}, hs, X, Y, S, nthr);
            net_rhs(tb, S, R, nthr, x, Y, F, K3);
            dp5_stage_input<3>({dp5::A41, dp5::A42, dp5::A43}, {K1, K2, K3}, hs, X, Y, S, nthr);
            net_rhs(tb, S, R, nthr, x, Y, F, K4);
            dp5_stage_input<4>({dp5::A51, dp5::A52, dp5::A53, dp5::A54}, {K1, K2, K3, K4}, hs, X, Y, S, nthr);
            net_rhs(tb, S, R, nthr, x, Y, F, K5);
            dp5_stage_input<5>({dp5::A61, dp5::A62, dp5::A63, dp5::A64, dp5::A65}, {K1, K2, K3, K4, K5}, hs, X, Y, S, nthr);
            net_rhs(tb, S, R, nthr, x, Y, F, K6);
            dp5_stage_input<5>({dp5::A71, dp5::A73, dp5::A74, dp5::A75, dp5::A76}, {K1, K3, K4, K5, K6}, hs, X, Y, S, nthr);
            double *K7 = K2;
            net_rhs(tb, S, R, nthr, x, Y, F, K7);
            double q = 0.0;
            for (int sp = 0; sp < S; ++sp) {
                const int v = sp * nthr;
                double e = fma(dp5::E1, K1[v], 0.0);
                e = fma(dp5::E3, K3[v], e);
                e = fma(dp5::E4, K4[v], e);
                e = fma(dp5::E5, K5[v], e);
                e = fma(dp5::E6, K6[v], e);
                e = fma(dp5::E7, K7[v], e);
                const double sc = fma(rtol, fmax(fabs(X[v]), fabs(Y[v])), atol);
                const double r = __ddiv_rn(__dmul_rn(hs, e), sc);
                q = fma(r, r, q);
            }
            const double err = __dsqrt_rn(__ddiv_rn(q, (double)S));
            const double fac_max = after_reject ? 1.0 : 5.0;
            const double fac = err == 0.0 ? fac_max
                               : isfinite(err) ? fmin(fac_max, fmax(0.2, __ddiv_rn(0.9, __dsqrt_rn(__dsqrt_rn(err)))))
                                               : 0.2;
            if (err <= 1.0) {
                ++accepted;
                t = clip ? to : __dadd_rn(t, hs);
                double *old = X;
                X = Y;
                Y = old;
                k1 = 1 - k1;
                after_reject = false;
                if (clip) {
                    net_observe(ot, L, nthr, X, out + m * L);
                    ++m;
                }
            } else {
                after_reject = true;
            }
            h = __dmul_rn(hs, fac);
        }
    }
    if (stats) net_add_stats(stats, valid, attempts, accepted, failed);
}

// ---------------------------------------------------------------------------------------------------------------------
// Adaptive Rosenbrock Rodas3 (VS_OBJ_MASS_ACTION_STIFF): the work split, tables, output times and counts of
// network_adaptive_kernel, plus the stiff tables (Jacobian scatter list and elimination program, stiff_program) in shared
// memory.  Per-trajectory state, [variable][thread]:
//   x[k], X[S] the state at t, fX[S] = f(X) (kept across rejected attempts), Y[S] the stage input and then the new
//   solution, K[4][S] the stages (each right-hand side is formed in its K slot and solved in place), F[R] the fluxes,
//   LU[nlu] the factor of G = I/(h gamma) - J(X), one slot per nonzero of L+U.
// Every index into the tables is warp-uniform, so each table read is a broadcast.  Nothing touches global memory inside the
// step loop but the observables written at output times.
// ---------------------------------------------------------------------------------------------------------------------
namespace rodas3 {   // Sandu et al. 1997 (as in KPP's Rosenbrock.f90), autonomous form; each the correctly rounded double
constexpr double GAMMA = 0.5;
constexpr double C21 = 4.0, C31 = 1.0, C32 = -1.0, C41 = 1.0, C42 = -1.0, C43 = -8.0 / 3.0;
}  // namespace rodas3

struct NetStiffTables {
    const int *jptr, *jcol, *jtp, *jt;     // Jacobian scatter
    const int *ord, *piv;                  // elimination order, pivot slots
    const int *lptr, *lent, *uptr, *uent;  // L columns and U rows: slot*128 + species
    const int *upd;                        // update targets
};

__device__ __forceinline__ NetStiffTables net_load_stiff(double *smem, const NetDev &net) {
    const NetLayout &n = net.n;
    const int S = n.S, R = n.R, nthr = blockDim.x, tid = threadIdx.x;
    int *base = reinterpret_cast<int *>(smem + net_adaptive_table_bytes(n) / sizeof(double));
    const int len = 4 * S + R + 4 + 2 * n.ncol + n.njt + n.nlow + n.nup + n.nupd;
    for (int e = tid; e < len; e += nthr) base[e] = (int)net.tab[n.o_stiff + e];
    NetStiffTables t;
    t.jptr = base;
    t.jcol = t.jptr + R + 1;
    t.jtp = t.jcol + n.ncol;
    t.jt = t.jtp + n.ncol + 1;
    t.ord = t.jt + n.njt;
    t.piv = t.ord + S;
    t.lptr = t.piv + S;
    t.lent = t.lptr + S + 1;
    t.uptr = t.lent + n.nlow;
    t.uent = t.uptr + S + 1;
    t.upd = t.uent + n.nup;
    return t;
}

// d(side product)/dX_c of a reaction side (a, b) (a one-species side in slot a)
__device__ __forceinline__ double net_dside(int a, int b, int c, const double *Y, int nthr) {
    if (a < 0) return 0.0;
    if (b < 0) return a == c ? 1.0 : 0.0;
    if (a == c) return b == c ? __dmul_rn(2.0, Y[c * nthr]) : Y[b * nthr];
    return b == c ? Y[a * nthr] : 0.0;
}

// LU = the factor of I/(hs gamma) - J(X), assembled and factored in program order.  false: a zero or non-finite pivot.
__device__ __forceinline__ bool net_factor(const NetTables &tb, const NetStiffTables &st, const NetLayout &n, int nthr,
                                           const double *x, const double *X, double ghinv, double *LU) {
    for (int e = 0; e < n.nlu; ++e) LU[e * nthr] = 0.0;
    for (int r = 0; r < n.R; ++r) {
        const int e1 = st.jptr[r + 1];
        int e = st.jptr[r];
        if (e == e1) continue;
        const int4 sp = tb.ri[r];
        const int2 cc = tb.rc[r];
        const double2 kc = tb.rk[r];
        const double kf = cc.x >= 0 ? x[cc.x * nthr] : kc.x;
        const bool rev = cc.y != NET_IRREV;
        const double kr = rev ? (cc.y >= 0 ? x[cc.y * nthr] : kc.y) : 0.0;
        for (; e < e1; ++e) {
            const int c = st.jcol[e];
            const double dpf = net_dside(sp.x, sp.y, c, X, nthr);
            const double d = rev ? fma(kf, dpf, -__dmul_rn(kr, net_dside(sp.z, sp.w, c, X, nthr))) : __dmul_rn(kf, dpf);
            for (int u = st.jtp[e]; u < st.jtp[e + 1]; ++u) {
                const int code = st.jt[u];
                double *a = LU + (code >> 3) * nthr;
                *a = fma(-(double)((code & 7) - 2), d, *a);
            }
        }
    }
    for (int p = 0; p < n.S; ++p) LU[st.piv[p] * nthr] = __dadd_rn(LU[st.piv[p] * nthr], ghinv);
    int u = 0;
    for (int p = 0; p < n.S; ++p) {
        const double pv = LU[st.piv[p] * nthr];
        if (!(pv != 0.0 && isfinite(pv))) return false;
        const int u0 = st.uptr[p], u1 = st.uptr[p + 1];
        for (int e = st.lptr[p]; e < st.lptr[p + 1]; ++e) {
            double *lp = LU + (st.lent[e] >> 7) * nthr;
            const double l = __ddiv_rn(*lp, pv);
            *lp = l;
            for (int f = u0; f < u1; ++f, ++u) {
                double *a = LU + st.upd[u] * nthr;
                *a = fma(-l, LU[(st.uent[f] >> 7) * nthr], *a);
            }
        }
    }
    return true;
}

// b = G^{-1} b in place: forward substitution with the unit lower factor by columns, back substitution by rows.
__device__ __forceinline__ void net_solve(const NetStiffTables &st, int S, int nthr, const double *LU, double *b) {
    for (int p = 0; p < S; ++p) {
        const double bp = b[st.ord[p] * nthr];
        for (int e = st.lptr[p]; e < st.lptr[p + 1]; ++e) {
            const int code = st.lent[e];
            double *bi = b + (code & 127) * nthr;
            *bi = fma(-LU[(code >> 7) * nthr], bp, *bi);
        }
    }
    for (int p = S - 1; p >= 0; --p) {
        double acc = b[st.ord[p] * nthr];
        for (int e = st.uptr[p]; e < st.uptr[p + 1]; ++e) {
            const int code = st.uent[e];
            acc = fma(-LU[(code >> 7) * nthr], b[(code & 127) * nthr], acc);
        }
        b[st.ord[p] * nthr] = __ddiv_rn(acc, LU[st.piv[p] * nthr]);
    }
}

// The cube root of a in [1e-3, 1e3] by correctly rounded operations only: a fixed bit-level first guess, then four Newton
// steps y = (2y + a/y^2) / 3.  The oracle restates it (ma_cbrt), so the step-size sequence is the same bits on both.
__device__ __forceinline__ double net_cbrt(double a) {
    double y = __longlong_as_double((long long)((unsigned long long)__double_as_longlong(a) / 3ull + 0x2A9F7893782DA1CEull));
#pragma unroll
    for (int i = 0; i < 4; ++i) y = __ddiv_rn(fma(2.0, y, __ddiv_rn(a, __dmul_rn(y, y))), 3.0);
    return y;
}

__global__ void __launch_bounds__(NET_THREADS) network_rosenbrock_kernel(int k, SourceDev src, ScaleDev s, NetDev net,
                                                                         uint64_t i_begin, uint64_t i_end,
                                                                         double *__restrict__ fvals,
                                                                         unsigned long long *__restrict__ stats) {
    extern __shared__ __align__(16) double smem[];
    const NetLayout &n = net.n;
    const int S = n.S, R = n.R, L = n.L, NT = n.NT, nthr = blockDim.x, tid = threadIdx.x;
    const NetTables tb = net_load_tables(smem, net);
    const NetOutputs ot = net_load_outputs(smem, net);
    const NetStiffTables st = net_load_stiff(smem, net);
    __syncthreads();
    const uint64_t rows = i_end - i_begin;
    const uint64_t row = (uint64_t)blockIdx.x * nthr + tid;
    const bool valid = row < rows;                                 // every lane stays for the warp reduction of the counts
    unsigned attempts = 0, accepted = 0;
    bool failed = false;
    if (valid) {
        double *x = smem + net_stiff_table_bytes(n) / sizeof(double) + tid;
        const size_t sl = (size_t)S * nthr;
        double *X = x + (size_t)k * nthr, *fX = X + sl, *Y = fX + sl, *K1 = Y + sl, *K2 = K1 + sl, *K3 = K2 + sl, *K4 = K3 + sl;
        double *F = K4 + sl, *LU = F + (size_t)R * nthr;
        const int p = blockIdx.y;
        net_point(k, src, s, net, i_begin + row, p, x, X, nthr);
        double *out = fvals + ((uint64_t)p * rows + row) * (uint64_t)(L * NT);
        const double rtol = n.rtol, atol = n.atol;
        const unsigned max_steps = (unsigned)n.max_steps;
        net_rhs(tb, S, R, nthr, x, X, F, fX);
        double t = 0.0, h = n.h0;
        bool after_reject = false;
        for (int m = 0; m < NT;) {
            const double to = ot.tout[m];
            double hs;
            bool clip;
            if (!net_next_step(t, h, to, attempts, max_steps, m, L, NT, out, hs, clip)) {
                failed = true;
                break;
            }
            ++attempts;
            if (!net_factor(tb, st, n, nthr, x, X, __ddiv_rn(1.0, __dmul_rn(rodas3::GAMMA, hs)), LU)) {
                after_reject = true;                               // singular: reject, the trajectory goes on
                h = __dmul_rn(hs, 0.2);
                continue;
            }
            const double c21 = __ddiv_rn(rodas3::C21, hs), c31 = __ddiv_rn(rodas3::C31, hs), c32 = __ddiv_rn(rodas3::C32, hs),
                         c41 = __ddiv_rn(rodas3::C41, hs), c42 = __ddiv_rn(rodas3::C42, hs), c43 = __ddiv_rn(rodas3::C43, hs);
            for (int sp = 0; sp < S; ++sp) K1[sp * nthr] = fX[sp * nthr];
            net_solve(st, S, nthr, LU, K1);
            for (int sp = 0; sp < S; ++sp) K2[sp * nthr] = fma(c21, K1[sp * nthr], fX[sp * nthr]);
            net_solve(st, S, nthr, LU, K2);
            for (int sp = 0; sp < S; ++sp) Y[sp * nthr] = fma(2.0, K1[sp * nthr], X[sp * nthr]);
            net_rhs(tb, S, R, nthr, x, Y, F, K3);
            for (int sp = 0; sp < S; ++sp) {
                const int v = sp * nthr;
                K3[v] = fma(c32, K2[v], fma(c31, K1[v], K3[v]));
            }
            net_solve(st, S, nthr, LU, K3);
            for (int sp = 0; sp < S; ++sp) Y[sp * nthr] = __dadd_rn(Y[sp * nthr], K3[sp * nthr]);
            net_rhs(tb, S, R, nthr, x, Y, F, K4);
            for (int sp = 0; sp < S; ++sp) {
                const int v = sp * nthr;
                K4[v] = fma(c43, K3[v], fma(c42, K2[v], fma(c41, K1[v], K4[v])));
            }
            net_solve(st, S, nthr, LU, K4);
            double q = 0.0;
            for (int sp = 0; sp < S; ++sp) {
                const int v = sp * nthr;
                const double y = __dadd_rn(Y[v], K4[v]);
                Y[v] = y;
                const double sc = fma(rtol, fmax(fabs(X[v]), fabs(y)), atol);
                const double r = __ddiv_rn(K4[v], sc);
                q = fma(r, r, q);
            }
            const double err = __dsqrt_rn(__ddiv_rn(q, (double)S));
            const double fac_max = after_reject ? 1.0 : 6.0;
            const double fac = isfinite(err) ? fmin(fac_max, fmax(0.2, __ddiv_rn(0.9, net_cbrt(fmin(fmax(err, 1e-3), 1e3))))) : 0.2;
            if (err <= 1.0) {
                ++accepted;
                t = clip ? to : __dadd_rn(t, hs);
                double *old = X;
                X = Y;
                Y = old;
                after_reject = false;
                if (clip) {
                    net_observe(ot, L, nthr, X, out + m * L);
                    ++m;
                }
                if (m < NT) net_rhs(tb, S, R, nthr, x, X, F, fX);
            } else {
                after_reject = true;
            }
            h = __dmul_rn(hs, fac);
        }
    }
    if (stats) net_add_stats(stats, valid, attempts, accepted, failed);
}

int network_check_fit(vs_ctx *c, int k, const ObjectiveDev &o) {
    const NetLayout n = net_layout(o.host, o.id);
    VS_REQUIRE(!n.stiff || net_smem(n, k, 32) <= c->smem_optin, VS_ERR_UNSUPPORTED,
               "stiff mass-action network with k=%d, S=%d, R=%d and nnz(LU) = %d factor nonzeros needs %zu bytes of shared memory "
               "for 32 trajectories, the device has %zu", k, n.S, n.R, n.nlu, net_smem(n, k, 32), c->smem_optin);
    VS_REQUIRE(net_smem(n, k, 32) <= c->smem_optin, VS_ERR_UNSUPPORTED,
               "mass-action network with k=%d, S=%d, R=%d needs %zu bytes of shared memory for 32 trajectories, the device has %zu",
               k, n.S, n.R, net_smem(n, k, 32), c->smem_optin);
    return VS_OK;
}

int launch_network_values(vs_ctx *c, int k, const SourceDev &src, const ScaleDev &s, const ObjectiveDev &o, uint64_t i_begin,
                          uint64_t i_end, double *fvals, bool count) {
    VS_TRY(network_check_fit(c, k, o));
    const uint64_t rows = i_end - i_begin;
    if (rows == 0) return VS_OK;
    NetDev net{o.params, net_layout(o.host, o.id)};
    const bool adaptive = net.n.NT > 0;                 // adaptive or stiff
    unsigned long long *stats = nullptr;
    if (adaptive && count) {                          // vs_last_network_stats: the counts of this call only
        VS_TRY(ensure(c, c->stats_buf, 4 * sizeof(unsigned long long)));
        stats = (unsigned long long *)c->stats_buf.p;
        VS_CUDA(cudaMemsetAsync(stats, 0, 4 * sizeof(unsigned long long), c->stream));
    }
    const int nthr = net_smem(net.n, k, NET_THREADS) <= c->smem_optin ? NET_THREADS : 32;
    const size_t smem = net_smem(net.n, k, nthr);
    dim3 grid((unsigned)((rows + nthr - 1) / nthr), (unsigned)(2 + 2 * k));
    const char *name = net.n.stiff ? "network_rosenbrock_kernel" : adaptive ? "network_adaptive_kernel" : "network_values_kernel";
    if (net.n.stiff) {
        VS_CUDA(cudaFuncSetAttribute(network_rosenbrock_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        time_begin(c);
        network_rosenbrock_kernel<<<grid, nthr, smem, c->stream>>>(k, src, s, net, i_begin, i_end, fvals, stats);
    } else if (adaptive) {
        VS_CUDA(cudaFuncSetAttribute(network_adaptive_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        time_begin(c);
        network_adaptive_kernel<<<grid, nthr, smem, c->stream>>>(k, src, s, net, i_begin, i_end, fvals, stats);
    } else {
        VS_CUDA(cudaFuncSetAttribute(network_values_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        time_begin(c);
        network_values_kernel<<<grid, nthr, smem, c->stream>>>(k, src, s, net, i_begin, i_end, fvals);
    }
    time_end(c);
    c->launches++;
    VS_CUDA(cudaGetLastError());
    if (!c->opt.trace.empty()) {                      // VS_TRACE: the form that ran (64 or 32 trajectories per CTA) and its grid
        if (FILE *fp = fopen(c->opt.trace.c_str(), "a")) {
            fprintf(fp, "# %s nthr=%d gx=%u gy=%u smem=%zu rows=%llu\n", name, nthr, grid.x, grid.y, smem, (unsigned long long)rows);
            fclose(fp);
        }
    }
    return VS_OK;
}

}  // namespace vs
