/* CPU restatement of the mass-action network objectives (VS_OBJ_MASS_ACTION, VS_OBJ_MASS_ACTION_ADAPTIVE).
 *
 * TEST INFRASTRUCTURE ONLY (oracle/__init__.py), never linked into libvarsens_b200.so.  oracle/Makefile builds it into
 * liboracle.so (-ffp-contract=off: the fma() calls below are the only fused operations); oracle/mass_action.py feeds it the
 * sample points of oracle/oracle.c's orc_sample_flat, so the values belong to the same design as orc_values'.
 */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

/* Mass-action reaction network (layout in include/varsens_b200.h), FROZEN ARITHMETIC shared with the device kernels
 * (varsens_b200/csrc/device.cuh: MassAction, MassActionAdaptive):
 *   P = 1.0 (no species on the side), X[s0] (one), X[s0] * X[s1] (two; a side given as (-1, s) is the one-species side s)
 *   flux_r = fma(kf, Pf, -(kr * Pr))   reversible;   flux_r = kf * Pf   irreversible (kr_coord = -1 and kr_const = 0)
 *   d_s = 0.0, then in ascending reaction order over the net coefficients c != 0 of species s (products - reactants):
 *         c = +1: d + flux   c = -1: d - flux   |c| = 2: fma(c, flux, d)
 *   fixed step: stages and update exactly those of oracle.c's f_rk4_chain;  observable o = fma(w, X_s, acc) from 0.0 over the
 *   nonzero w[o][s], ascending s.
 * The chain X_0 <-> ... <-> X_S written as a fixed-step network reproduces oracle.c's f_rk4_chain bit for bit. */
#define ORC_MA_MAXS 128
#define ORC_MA_MAXR 512
#define MA_HDR 5                /* S R L dt nsteps */
#define MA_ADAPTIVE_HDR 8       /* S R L NT rtol atol h0 max_steps */

static double ma_side(const double *Y, double s0, double s1) {
    int a = (int)s0, b = (int)s1;
    if (a < 0) { a = b; b = -1; }
    if (a < 0) return 1.0;
    if (b < 0) return Y[a];
    return Y[a] * Y[b];
}

static double ma_coef(const double *q, int s) {
    return (double)(((int)q[2] == s) + ((int)q[3] == s) - ((int)q[0] == s) - ((int)q[1] == s));
}

/* rec: the R reaction records of 8 doubles each. */
static void ma_rhs(const double *rec, int S, int R, const double *x, const double *Y, double *flux, double *d) {
    for (int r = 0; r < R; ++r) {
        const double *q = rec + 8 * r;
        double kf = q[4] >= 0 ? x[(int)q[4]] : q[5];
        double pf = ma_side(Y, q[0], q[1]);
        if (q[6] < 0 && q[7] == 0.0) {
            flux[r] = kf * pf;
        } else {
            double kr = q[6] >= 0 ? x[(int)q[6]] : q[7];
            double back = kr * ma_side(Y, q[2], q[3]);
            flux[r] = fma(kf, pf, -back);
        }
    }
    for (int s = 0; s < S; ++s) {
        double acc = 0.0;
        for (int r = 0; r < R; ++r) {
            double c = ma_coef(rec + 8 * r, s);
            if (c == 1.0) acc = acc + flux[r];
            else if (c == -1.0) acc = acc - flux[r];
            else if (c != 0.0) acc = fma(c, flux[r], acc);
        }
        d[s] = acc;
    }
}

static void ma_observe(const double *w, int S, int L, const double *X, double *out) {
    for (int o = 0; o < L; ++o) {
        double acc = 0.0;
        for (int s = 0; s < S; ++s)
            if (w[o * S + s] != 0.0) acc = fma(w[o * S + s], X[s], acc);
        out[o] = acc;
    }
}

static void f_mass_action(const double *x, const double *par, double *out) {
    int S = (int)par[0], R = (int)par[1], L = (int)par[2], nsteps = (int)par[4];
    double dt = par[3];
    double h2 = 0.5 * dt, h6 = dt / 6.0;
    double X[ORC_MA_MAXS], T[ORC_MA_MAXS], a[ORC_MA_MAXS], d[ORC_MA_MAXS], flux[ORC_MA_MAXR];
    const double *rec = par + MA_HDR, *init = rec + 8 * R, *w = init + 2 * S;
    for (int s = 0; s < S; ++s) X[s] = init[2 * s] >= 0 ? x[(int)init[2 * s]] : init[2 * s + 1];
    for (int it = 0; it < nsteps; ++it) {
        ma_rhs(rec, S, R, x, X, flux, d);
        for (int s = 0; s < S; ++s) { a[s] = d[s]; T[s] = fma(h2, d[s], X[s]); }
        ma_rhs(rec, S, R, x, T, flux, d);
        for (int s = 0; s < S; ++s) { a[s] = fma(2.0, d[s], a[s]); T[s] = fma(h2, d[s], X[s]); }
        ma_rhs(rec, S, R, x, T, flux, d);
        for (int s = 0; s < S; ++s) { a[s] = fma(2.0, d[s], a[s]); T[s] = fma(dt, d[s], X[s]); }
        ma_rhs(rec, S, R, x, T, flux, d);
        for (int s = 0; s < S; ++s) { double t = a[s] + d[s]; X[s] = fma(h6, t, X[s]); }
    }
    ma_observe(w, S, L, X, out);
}

/* Adaptive stepper: the frozen arithmetic of varsens_b200/csrc/device.cuh: MassActionAdaptive, bit for bit.
 * Dormand-Prince 5(4), Hairer-Norsett-Wanner I, Table 5.2: a[i][j] of stage i+2 (row 5 = b), e_j = b_j - bhat_j. */
static const double A[6][6] = {
    {1.0 / 5.0},
    {3.0 / 40.0, 9.0 / 40.0},
    {44.0 / 45.0, -56.0 / 15.0, 32.0 / 9.0},
    {19372.0 / 6561.0, -25360.0 / 2187.0, 64448.0 / 6561.0, -212.0 / 729.0},
    {9017.0 / 3168.0, -355.0 / 33.0, 46732.0 / 5247.0, 49.0 / 176.0, -5103.0 / 18656.0},
    {35.0 / 384.0, 0.0, 500.0 / 1113.0, 125.0 / 192.0, -2187.0 / 6784.0, 11.0 / 84.0},
};
static const double E[7] = {71.0 / 57600.0, 0.0, -71.0 / 16695.0, 71.0 / 1920.0, -17253.0 / 339200.0, 22.0 / 525.0, -1.0 / 40.0};

/* out[m*L + o]: observable o at time t_{m+1}; info = {attempts, accepted, failed}. */
static void f_mass_action_adaptive(const double *x, const double *par, double *out, int64_t *info) {
    int S = (int)par[0], R = (int)par[1], L = (int)par[2], NT = (int)par[3];
    double rtol = par[4], atol = par[5], h = par[6];
    int64_t max_steps = (int64_t)par[7];
    const double *rec = par + MA_ADAPTIVE_HDR, *init = rec + 8 * R, *w = init + 2 * S, *times = w + L * S;
    double X[ORC_MA_MAXS], Y[ORC_MA_MAXS], K[7][ORC_MA_MAXS], flux[ORC_MA_MAXR];
    int64_t attempts = 0, accepted = 0, failed = 0;
    for (int s = 0; s < S; ++s) X[s] = init[2 * s] >= 0 ? x[(int)init[2 * s]] : init[2 * s + 1];
    ma_rhs(rec, S, R, x, X, flux, K[0]);
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
        for (int i = 1; i <= 6; ++i) {            /* stages 2..7 into K[1..6] (K[6] = K7) */
            for (int s = 0; s < S; ++s) {
                double acc = 0.0;
                for (int j = 0; j < i; ++j)
                    if (A[i - 1][j] != 0.0) acc = fma(A[i - 1][j], K[j][s], acc);
                Y[s] = fma(hs, acc, X[s]);
            }
            ma_rhs(rec, S, R, x, Y, flux, K[i]);
        }
        double q = 0.0;
        for (int s = 0; s < S; ++s) {
            double e = 0.0;
            for (int j = 0; j < 7; ++j)
                if (E[j] != 0.0) e = fma(E[j], K[j][s], e);
            double sc = fma(rtol, fmax(fabs(X[s]), fabs(Y[s])), atol);
            double r = (hs * e) / sc;
            q = fma(r, r, q);
        }
        double err = sqrt(q / (double)S);
        double fac_max = after_reject ? 1.0 : 5.0;
        double fac = err == 0.0 ? fac_max : isfinite(err) ? fmin(fac_max, fmax(0.2, 0.9 / sqrt(sqrt(err)))) : 0.2;
        if (err <= 1.0) {
            ++accepted;
            t = clip ? to : t + hs;
            for (int s = 0; s < S; ++s) { X[s] = Y[s]; K[0][s] = K[6][s]; }
            after_reject = 0;
            if (clip) {
                ma_observe(w, S, L, X, out + m * L);
                ++m;
            }
        } else {
            after_reject = 1;
        }
        h = hs * fac;
    }
    info[0] = attempts;
    info[1] = accepted;
    info[2] = failed;
}

/* out[p*L + o], p < count: the L observables of the points x[p*k .. p*k+k). */
void ma_values(int k, uint64_t count, const double *x, const double *par, double *out) {
    int L = (int)par[2];
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t p = 0; p < (int64_t)count; ++p) f_mass_action(x + (size_t)p * k, par, out + (size_t)p * L);
}

/* out[p*L*NT + c], info[p*3 + i], p < count: the points x[p*k .. p*k+k). */
void ma_values_adaptive(int k, uint64_t count, const double *x, const double *par, double *out, int64_t *info) {
    int l = (int)par[2] * (int)par[3];
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t p = 0; p < (int64_t)count; ++p)
        f_mass_action_adaptive(x + (size_t)p * k, par, out + (size_t)p * l, info + 3 * p);
}
