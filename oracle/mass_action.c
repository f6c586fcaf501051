/* CPU restatement of the mass-action network objective (VS_OBJ_MASS_ACTION).
 *
 * TEST INFRASTRUCTURE ONLY (oracle/__init__.py), never linked into libvarsens_b200.so.  oracle/mass_action.py compiles it
 * with the flags of oracle/Makefile (-ffp-contract=off: the fma() calls below are the only fused operations) and feeds it
 * the sample points of oracle/oracle.c's orc_sample_flat, so the values belong to the same design as orc_values'.
 */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

/* Mass-action reaction network (VS_OBJ_MASS_ACTION, layout in include/varsens_b200.h), FROZEN ARITHMETIC shared with the
 * device kernel (varsens_b200/csrc/device.cuh: MassAction):
 *   P = 1.0 (no species on the side), X[s0] (one), X[s0] * X[s1] (two; a side given as (-1, s) is the one-species side s)
 *   flux_r = fma(kf, Pf, -(kr * Pr))   reversible;   flux_r = kf * Pf   irreversible (kr_coord = -1 and kr_const = 0)
 *   d_s = 0.0, then in ascending reaction order over the net coefficients c != 0 of species s (products - reactants):
 *         c = +1: d + flux   c = -1: d - flux   |c| = 2: fma(c, flux, d)
 *   stages and update exactly those of oracle.c's f_rk4_chain;  observable o = fma(w, X_s, acc) from 0.0 over the nonzero w[o][s],
 *   ascending s.
 * The chain X_0 <-> ... <-> X_S written as a network reproduces oracle.c's f_rk4_chain bit for bit. */
#define ORC_MA_MAXS 128
#define ORC_MA_MAXR 512

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

static void ma_rhs(const double *par, const double *x, const double *Y, double *flux, double *d) {
    int S = (int)par[0], R = (int)par[1];
    for (int r = 0; r < R; ++r) {
        const double *q = par + 5 + 8 * r;
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
            double c = ma_coef(par + 5 + 8 * r, s);
            if (c == 1.0) acc = acc + flux[r];
            else if (c == -1.0) acc = acc - flux[r];
            else if (c != 0.0) acc = fma(c, flux[r], acc);
        }
        d[s] = acc;
    }
}

static void f_mass_action(const double *x, const double *par, double *out) {
    int S = (int)par[0], R = (int)par[1], L = (int)par[2], nsteps = (int)par[4];
    double dt = par[3];
    double h2 = 0.5 * dt, h6 = dt / 6.0;
    double X[ORC_MA_MAXS], T[ORC_MA_MAXS], a[ORC_MA_MAXS], d[ORC_MA_MAXS], flux[ORC_MA_MAXR];
    const double *init = par + 5 + 8 * R, *w = init + 2 * S;
    for (int s = 0; s < S; ++s) X[s] = init[2 * s] >= 0 ? x[(int)init[2 * s]] : init[2 * s + 1];
    for (int it = 0; it < nsteps; ++it) {
        ma_rhs(par, x, X, flux, d);
        for (int s = 0; s < S; ++s) { a[s] = d[s]; T[s] = fma(h2, d[s], X[s]); }
        ma_rhs(par, x, T, flux, d);
        for (int s = 0; s < S; ++s) { a[s] = fma(2.0, d[s], a[s]); T[s] = fma(h2, d[s], X[s]); }
        ma_rhs(par, x, T, flux, d);
        for (int s = 0; s < S; ++s) { a[s] = fma(2.0, d[s], a[s]); T[s] = fma(dt, d[s], X[s]); }
        ma_rhs(par, x, T, flux, d);
        for (int s = 0; s < S; ++s) { double t = a[s] + d[s]; X[s] = fma(h6, t, X[s]); }
    }
    for (int o = 0; o < L; ++o) {
        double acc = 0.0;
        for (int s = 0; s < S; ++s)
            if (w[o * S + s] != 0.0) acc = fma(w[o * S + s], X[s], acc);
        out[o] = acc;
    }
}

/* out[p*L + o], p < count: the L observables of the points x[p*k .. p*k+k). */
void ma_values(int k, uint64_t count, const double *x, const double *par, double *out) {
    int L = (int)par[2];
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t p = 0; p < (int64_t)count; ++p) f_mass_action(x + (size_t)p * k, par, out + (size_t)p * L);
}
