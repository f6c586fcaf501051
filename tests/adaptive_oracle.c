/* CPU restatement of the adaptive mass-action network objective (VS_OBJ_MASS_ACTION_ADAPTIVE).
 *
 * TEST INFRASTRUCTURE ONLY, never linked into libvarsens_b200.so.  tests/adaptive_oracle.py compiles it with the flags of
 * oracle/Makefile (-ffp-contract=off: the fma() calls below are the only fused operations) and feeds it the sample points of
 * oracle.cport.sample_flat.  The right-hand side is oracle/mass_action.c's (f_mass_action) for the adaptive header; the
 * stepper restates the frozen arithmetic of varsens_b200/csrc/device.cuh: MassActionAdaptive bit for bit.
 */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

#define AD_MAXS 128
#define AD_MAXR 512
#define AD_HDR 8

static double ad_side(const double *Y, double s0, double s1) {
    int a = (int)s0, b = (int)s1;
    if (a < 0) { a = b; b = -1; }
    if (a < 0) return 1.0;
    if (b < 0) return Y[a];
    return Y[a] * Y[b];
}

static double ad_coef(const double *q, int s) {
    return (double)(((int)q[2] == s) + ((int)q[3] == s) - ((int)q[0] == s) - ((int)q[1] == s));
}

static void ad_rhs(const double *par, const double *x, const double *Y, double *flux, double *d) {
    int S = (int)par[0], R = (int)par[1];
    for (int r = 0; r < R; ++r) {
        const double *q = par + AD_HDR + 8 * r;
        double kf = q[4] >= 0 ? x[(int)q[4]] : q[5];
        double pf = ad_side(Y, q[0], q[1]);
        if (q[6] < 0 && q[7] == 0.0) {
            flux[r] = kf * pf;
        } else {
            double kr = q[6] >= 0 ? x[(int)q[6]] : q[7];
            double back = kr * ad_side(Y, q[2], q[3]);
            flux[r] = fma(kf, pf, -back);
        }
    }
    for (int s = 0; s < S; ++s) {
        double acc = 0.0;
        for (int r = 0; r < R; ++r) {
            double c = ad_coef(par + AD_HDR + 8 * r, s);
            if (c == 1.0) acc = acc + flux[r];
            else if (c == -1.0) acc = acc - flux[r];
            else if (c != 0.0) acc = fma(c, flux[r], acc);
        }
        d[s] = acc;
    }
}

/* Dormand-Prince 5(4), Hairer-Norsett-Wanner I, Table 5.2: a[i][j] of stage i+2 (row 5 = b), e_j = b_j - bhat_j. */
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
    const double *init = par + AD_HDR + 8 * R, *w = init + 2 * S, *times = w + L * S;
    double X[AD_MAXS], Y[AD_MAXS], K[7][AD_MAXS], flux[AD_MAXR];
    int64_t attempts = 0, accepted = 0, failed = 0;
    for (int s = 0; s < S; ++s) X[s] = init[2 * s] >= 0 ? x[(int)init[2 * s]] : init[2 * s + 1];
    ad_rhs(par, x, X, flux, K[0]);
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
            ad_rhs(par, x, Y, flux, K[i]);
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
                for (int o = 0; o < L; ++o) {
                    double acc = 0.0;
                    for (int s = 0; s < S; ++s)
                        if (w[o * S + s] != 0.0) acc = fma(w[o * S + s], X[s], acc);
                    out[m * L + o] = acc;
                }
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

/* out[p*L*NT + c], info[p*3 + i], p < count: the points x[p*k .. p*k+k). */
void ad_values(int k, uint64_t count, const double *x, const double *par, double *out, int64_t *info) {
    int l = (int)par[2] * (int)par[3];
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t p = 0; p < (int64_t)count; ++p) f_mass_action_adaptive(x + (size_t)p * k, par, out + (size_t)p * l, info + 3 * p);
}
