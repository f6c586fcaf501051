/* CPU restatement of the stiff mass-action network objective (VS_OBJ_MASS_ACTION_STIFF: the description of
 * VS_OBJ_MASS_ACTION_ADAPTIVE integrated by Rodas3).
 *
 * TEST INFRASTRUCTURE ONLY (oracle/__init__.py), never linked into libvarsens_b200.so.  oracle/mass_action_stiff.py compiles
 * it into its own library with oracle/Makefile's flags (-ffp-contract=off: the fma() calls are the only fused operations).  It
 * includes oracle/mass_action.c, so the right-hand side (ma_rhs), the net coefficients (ma_coef) and the observable sum
 * (ma_observe) are the ones the fixed-step and Dormand-Prince restatements use.
 */
#include "mass_action.c"

#include <stdlib.h>
#include <string.h>

/* Stiff stepper: the frozen arithmetic of varsens_b200/csrc/device.cuh: MassActionStiff (Rodas3), bit for bit.  The factor's
 * pattern, the elimination order and the program are restated here on dense position-indexed arrays, independently of the
 * library's lists (kernels_network.cu: stiff_program). */

typedef struct {
    int S, nlu, ncol, njt;
    int ord[ORC_MA_MAXS];                    /* species at elimination position p */
    int pos[ORC_MA_MAXS];                    /* elimination position of species s */
    unsigned char F[ORC_MA_MAXS][ORC_MA_MAXS];   /* factor pattern, positions */
} MaStiff;

static int ma_reversible(const double *q) { return !(q[6] < 0 && q[7] == 0.0); }

/* species c is a column of reaction q: a reactant (a catalyst too), or a product of a reversible reaction */
static int ma_is_column(const double *q, int c) {
    return (int)q[0] == c || (int)q[1] == c || (ma_reversible(q) && ((int)q[2] == c || (int)q[3] == c));
}

static void ma_stiff_plan(const double *par, MaStiff *pl) {
    int S = (int)par[0], R = (int)par[1];
    const double *rec = par + MA_ADAPTIVE_HDR;
    static const unsigned char zero[ORC_MA_MAXS][ORC_MA_MAXS];
    unsigned char P[ORC_MA_MAXS][ORC_MA_MAXS], G[ORC_MA_MAXS][ORC_MA_MAXS], alive[ORC_MA_MAXS];
    memcpy(P, zero, sizeof P);
    memcpy(G, zero, sizeof G);
    pl->S = S;
    pl->ncol = pl->njt = 0;
    for (int s = 0; s < S; ++s) P[s][s] = 1;
    for (int r = 0; r < R; ++r) {
        const double *q = rec + 8 * r;
        for (int c = 0; c < S; ++c) {
            if (!ma_is_column(q, c)) continue;
            ++pl->ncol;
            for (int s = 0; s < S; ++s)
                if (ma_coef(q, s) != 0.0) { P[s][c] = 1; ++pl->njt; }
        }
    }
    for (int a = 0; a < S; ++a) {
        alive[a] = 1;
        for (int b = 0; b < S; ++b) G[a][b] = a != b && (P[a][b] || P[b][a]);
    }
    for (int p = 0; p < S; ++p) {                /* minimum degree, ties to the lowest species */
        int best = -1, bd = 0;
        for (int v = 0; v < S; ++v) {
            if (!alive[v]) continue;
            int d = 0;
            for (int u = 0; u < S; ++u) d += alive[u] && G[v][u];
            if (best < 0 || d < bd) { best = v; bd = d; }
        }
        alive[best] = 0;
        for (int u = 0; u < S; ++u)
            for (int w = 0; w < S; ++w)
                if (u != w && alive[u] && alive[w] && G[best][u] && G[best][w]) G[u][w] = 1;
        pl->ord[p] = best;
        pl->pos[best] = p;
    }
    pl->nlu = 0;
    for (int i = 0; i < S; ++i)
        for (int j = 0; j < S; ++j) pl->F[i][j] = P[pl->ord[i]][pl->ord[j]];
    for (int p = 0; p < S; ++p)                  /* symbolic LU without pivoting */
        for (int i = p + 1; i < S; ++i)
            if (pl->F[i][p])
                for (int j = p + 1; j < S; ++j)
                    if (pl->F[p][j]) pl->F[i][j] = 1;
    for (int i = 0; i < S; ++i)
        for (int j = 0; j < S; ++j) pl->nlu += pl->F[i][j];
}

/* d(side product)/dY_c of the side (s0, s1), ma_side's convention */
static double ma_dside(const double *Y, double s0, double s1, int c) {
    int a = (int)s0, b = (int)s1;
    if (a < 0) { a = b; b = -1; }
    if (a < 0) return 0.0;
    if (b < 0) return a == c ? 1.0 : 0.0;
    if (a == c) return b == c ? 2.0 * Y[c] : Y[b];
    return b == c ? Y[a] : 0.0;
}

/* cube root of a in [1e-3, 1e3]: bit-level first guess, four Newton steps (device.cuh: MassActionStiff) */
static double ma_cbrt(double a) {
    uint64_t u;
    double y;
    memcpy(&u, &a, 8);
    u = u / 3u + 0x2A9F7893782DA1CEull;
    memcpy(&y, &u, 8);
    for (int i = 0; i < 4; ++i) y = fma(2.0, y, a / (y * y)) / 3.0;
    return y;
}

/* b = G^{-1} b with the factor a (positions) */
static void ma_lu_solve(const MaStiff *pl, const double *a, double *b) {
    int S = pl->S;
    for (int p = 0; p < S; ++p)
        for (int i = p + 1; i < S; ++i)
            if (pl->F[i][p]) b[pl->ord[i]] = fma(-a[i * S + p], b[pl->ord[p]], b[pl->ord[i]]);
    for (int p = S - 1; p >= 0; --p) {
        double acc = b[pl->ord[p]];
        for (int j = p + 1; j < S; ++j)
            if (pl->F[p][j]) acc = fma(-a[p * S + j], b[pl->ord[j]], acc);
        b[pl->ord[p]] = acc / a[p * S + p];
    }
}

/* out[m*L + o], info = {attempts, accepted, failed}: f_mass_action_adaptive's layout and trajectory rules */
static void f_mass_action_stiff(const double *x, const double *par, const MaStiff *pl, double *out, int64_t *info) {
    int S = (int)par[0], R = (int)par[1], L = (int)par[2], NT = (int)par[3];
    double rtol = par[4], atol = par[5], h = par[6];
    int64_t max_steps = (int64_t)par[7];
    const double *rec = par + MA_ADAPTIVE_HDR, *init = rec + 8 * R, *w = init + 2 * S, *times = w + L * S;
    double X[ORC_MA_MAXS], Y[ORC_MA_MAXS], fX[ORC_MA_MAXS], K[4][ORC_MA_MAXS], flux[ORC_MA_MAXR];
    double *a = malloc(sizeof(double) * S * S);
    int64_t attempts = 0, accepted = 0, failed = 0;
    for (int s = 0; s < S; ++s) X[s] = init[2 * s] >= 0 ? x[(int)init[2 * s]] : init[2 * s + 1];
    ma_rhs(rec, S, R, x, X, flux, fX);
    double t = 0.0;
    int after_reject = 0;
    for (int m = 0; m < NT;) {
        double to = times[m], hs = h;
        int clip = t + hs >= to;
        if (clip) hs = to - t;
        if (attempts == max_steps || t + hs == t) {
            for (int e = m * L; e < NT * L; ++e) out[e] = NAN;
            failed = 1;
            break;
        }
        ++attempts;
        /* G = I/(hs gamma) - J(X): zero, scatter -nu dflux/dX over ascending reactions, add the diagonal, factor */
        for (int i = 0; i < S; ++i)
            for (int j = 0; j < S; ++j)
                if (pl->F[i][j]) a[i * S + j] = 0.0;
        for (int r = 0; r < R; ++r) {
            const double *q = rec + 8 * r;
            int rev = ma_reversible(q);
            double kf = q[4] >= 0 ? x[(int)q[4]] : q[5];
            double kr = rev ? (q[6] >= 0 ? x[(int)q[6]] : q[7]) : 0.0;
            for (int c = 0; c < S; ++c) {
                if (!ma_is_column(q, c)) continue;
                double dpf = ma_dside(X, q[0], q[1], c);
                double d = rev ? fma(kf, dpf, -(kr * ma_dside(X, q[2], q[3], c))) : kf * dpf;
                for (int s = 0; s < S; ++s) {
                    double nu = ma_coef(q, s);
                    if (nu != 0.0) {
                        double *e = a + pl->pos[s] * S + pl->pos[c];
                        *e = fma(-nu, d, *e);
                    }
                }
            }
        }
        double ghinv = 1.0 / (0.5 * hs);
        for (int p = 0; p < S; ++p) a[p * S + p] = a[p * S + p] + ghinv;
        int singular = 0;
        for (int p = 0; p < S && !singular; ++p) {
            double pv = a[p * S + p];
            if (!(pv != 0.0 && isfinite(pv))) { singular = 1; break; }
            for (int i = p + 1; i < S; ++i) {
                if (!pl->F[i][p]) continue;
                double l = a[i * S + p] / pv;
                a[i * S + p] = l;
                for (int j = p + 1; j < S; ++j)
                    if (pl->F[p][j]) a[i * S + j] = fma(-l, a[p * S + j], a[i * S + j]);
            }
        }
        if (singular) {
            after_reject = 1;
            h = hs * 0.2;
            continue;
        }
        double c21 = 4.0 / hs, c31 = 1.0 / hs, c32 = -1.0 / hs, c41 = 1.0 / hs, c42 = -1.0 / hs, c43 = (-8.0 / 3.0) / hs;
        for (int s = 0; s < S; ++s) K[0][s] = fX[s];
        ma_lu_solve(pl, a, K[0]);
        for (int s = 0; s < S; ++s) K[1][s] = fma(c21, K[0][s], fX[s]);
        ma_lu_solve(pl, a, K[1]);
        for (int s = 0; s < S; ++s) Y[s] = fma(2.0, K[0][s], X[s]);
        ma_rhs(rec, S, R, x, Y, flux, K[2]);
        for (int s = 0; s < S; ++s) K[2][s] = fma(c32, K[1][s], fma(c31, K[0][s], K[2][s]));
        ma_lu_solve(pl, a, K[2]);
        for (int s = 0; s < S; ++s) Y[s] = Y[s] + K[2][s];
        ma_rhs(rec, S, R, x, Y, flux, K[3]);
        for (int s = 0; s < S; ++s) K[3][s] = fma(c43, K[2][s], fma(c42, K[1][s], fma(c41, K[0][s], K[3][s])));
        ma_lu_solve(pl, a, K[3]);
        double q = 0.0;
        for (int s = 0; s < S; ++s) {
            Y[s] = Y[s] + K[3][s];
            double sc = fma(rtol, fmax(fabs(X[s]), fabs(Y[s])), atol);
            double r = K[3][s] / sc;
            q = fma(r, r, q);
        }
        double err = sqrt(q / (double)S);
        double fac_max = after_reject ? 1.0 : 6.0;
        double fac = isfinite(err) ? fmin(fac_max, fmax(0.2, 0.9 / ma_cbrt(fmin(fmax(err, 1e-3), 1e3)))) : 0.2;
        if (err <= 1.0) {
            ++accepted;
            t = clip ? to : t + hs;
            for (int s = 0; s < S; ++s) X[s] = Y[s];
            after_reject = 0;
            if (clip) {
                ma_observe(w, S, L, X, out + m * L);
                ++m;
            }
            if (m < NT) ma_rhs(rec, S, R, x, X, flux, fX);
        } else {
            after_reject = 1;
        }
        h = hs * fac;
    }
    free(a);
    info[0] = attempts;
    info[1] = accepted;
    info[2] = failed;
}

/* ma_values_adaptive's layout for the stiff description */
void ma_values_stiff(int k, uint64_t count, const double *x, const double *par, double *out, int64_t *info) {
    int l = (int)par[2] * (int)par[3];
    MaStiff *pl = malloc(sizeof(MaStiff));
    ma_stiff_plan(par, pl);
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t p = 0; p < (int64_t)count; ++p)
        f_mass_action_stiff(x + (size_t)p * k, par, pl, out + (size_t)p * l, info + 3 * p);
    free(pl);
}

/* The factor's sizes of a stiff description: {nnz(L+U) with the diagonal, below-diagonal entries, above-diagonal entries,
 * update operations of the factorisation, Jacobian columns, Jacobian scatter targets}, and the elimination order. */
void ma_stiff_sizes(const double *par, int64_t *sizes, int64_t *ord) {
    MaStiff *pl = malloc(sizeof(MaStiff));
    ma_stiff_plan(par, pl);
    int S = pl->S;
    int64_t low = 0, up = 0, upd = 0;
    for (int p = 0; p < S; ++p) {
        int64_t lp = 0, upp = 0;
        for (int i = p + 1; i < S; ++i) lp += pl->F[i][p];
        for (int j = p + 1; j < S; ++j) upp += pl->F[p][j];
        low += lp;
        up += upp;
        upd += lp * upp;
    }
    sizes[0] = pl->nlu;
    sizes[1] = low;
    sizes[2] = up;
    sizes[3] = upd;
    sizes[4] = pl->ncol;
    sizes[5] = pl->njt;
    for (int p = 0; p < S; ++p) ord[p] = pl->ord[p];
    free(pl);
}
