"""Adaptive mass-action network objective (VS_OBJ_MASS_ACTION_ADAPTIVE, packed layout in include/varsens_b200.h).  TEST
INFRASTRUCTURE, next to the fixed-step oracle (oracle/mass_action.py), whose sample points and network builders it reuses.

* ``values_adaptive``: the C restatement (tests/adaptive_oracle.c, frozen arithmetic shared with the device kernel) on the
  design points of oracle.cport.sample_flat -- (2+2k, rows, L*NT) in the order fM_1, fM_2, fN_j[0..k), fN_nj[0..k), and
  the four step counts of vs_last_network_stats.
* ``adaptive_of``: any fixed-step description (oracle.mass_action.chain_network / random_network) as an adaptive one.
* ``numpy_rhs`` / ``solve_ivp_values``: a numpy right-hand side and a tight scipy.integrate.solve_ivp reference.
"""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy

from oracle import cport

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
HDR = 8
WARP = 32          # the kernel's warps: 32 consecutive rows of one design point


def lib():
    """The compiled restatement, built on first use into the temporary directory (the source tree may be read-only), keyed
    by the source's hash; the compiler flags of oracle/Makefile."""
    global _LIB
    if _LIB is None:
        src = os.path.join(_HERE, "adaptive_oracle.c")
        tag = hashlib.sha1(open(src, "rb").read()).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "varsens_oracle_ad_%d_%s.so" % (os.getuid(), tag))
        if not os.path.exists(so):
            tmp = "%s.%d.tmp" % (so, os.getpid())
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra",
                                   "-shared", "-o", tmp, src, "-lm"])
            os.replace(tmp, so)
        L = ctypes.CDLL(so)
        L.ad_values.argtypes = [ctypes.c_int, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                ctypes.c_void_p]
        _LIB = L
    return _LIB


def adaptive_of(packed, times, rtol=1e-6, atol=1e-9, h0=None, max_steps=100000):
    """The fixed-step description ``packed`` ([S, R, L, dt, nsteps] + records + initial amounts + weights) as an adaptive one
    with output times ``times``; h0 = None is 1e-6 * times[-1], as in AdaptiveMassActionNetwork."""
    par = numpy.asarray(packed, dtype=numpy.float64)
    times = numpy.atleast_1d(numpy.asarray(times, dtype=numpy.float64))
    h0 = 1e-6 * float(times[-1]) if h0 is None else float(h0)
    head = [par[0], par[1], par[2], float(times.size), float(rtol), float(atol), h0, float(max_steps)]
    return numpy.concatenate([head, par[5:], times])


def points_values(P, params):
    """(rows, k) points -> ((rows, L*NT) values, (rows, 3) int64 {attempts, accepted, failed})."""
    par = numpy.ascontiguousarray(params, dtype=numpy.float64)
    P = numpy.ascontiguousarray(numpy.atleast_2d(P), dtype=numpy.float64)
    l = int(par[2]) * int(par[3])
    out = numpy.empty((P.shape[0], l))
    info = numpy.empty((P.shape[0], 3), dtype=numpy.int64)
    lib().ad_values(int(P.shape[1]), int(P.shape[0]), P.ctypes.data_as(ctypes.c_void_p), par.ctypes.data_as(ctypes.c_void_p),
                    out.ctypes.data_as(ctypes.c_void_p), info.ctypes.data_as(ctypes.c_void_p))
    return out, info


def values_adaptive(k, n, params, discard=0, scale=None, i0=0, i1=None, perm=None, raw=None):
    """((2+2k, i1-i0, L*NT) observables, stats) of base rows [i0,i1): the arguments of oracle.mass_action.values.  stats =
    [accepted, rejected, failed, lane work] over these rows, lane work = the sum over warps of (rows in the warp x the most
    attempts of any lane in it)."""
    i1 = n if i1 is None else i1
    rows = int(i1 - i0)
    pts = numpy.concatenate([cport.sample_flat(k, n, discard, scale, t * n + i0, t * n + i1, perm, raw)
                             for t in range(2 + 2 * k)], axis=0)
    out, info = points_values(pts, params)
    att = info[:, 0].reshape(2 + 2 * k, rows)
    work = 0
    for w0 in range(0, rows, WARP):
        w = att[:, w0:w0 + WARP]
        work += int(w.shape[1]) * int(w.max(axis=1).sum())
    acc = int(info[:, 1].sum())
    stats = numpy.array([acc, int(info[:, 0].sum()) - acc, int(info[:, 2].sum()), work], dtype=numpy.uint64)
    return out.reshape(2 + 2 * k, rows, -1), stats


def numpy_rhs(params, x):
    """f(t, y) of the adaptive description ``params`` at the scaled point x, for solve_ivp, and y(0)."""
    par = numpy.asarray(params, dtype=numpy.float64)
    x = numpy.asarray(x, dtype=numpy.float64)
    S, R = int(par[0]), int(par[1])
    rec = par[HDR:HDR + 8 * R].reshape(R, 8)
    init = par[HDR + 8 * R:HDR + 8 * R + 2 * S].reshape(S, 2)
    val = lambda c, v: x[int(c)] if c >= 0 else v                   # noqa: E731
    kf = numpy.array([val(q[4], q[5]) for q in rec])
    kr = numpy.array([val(q[6], q[7]) for q in rec])
    a = [[int(s) for s in q[0:2] if s >= 0] for q in rec]
    b = [[int(s) for s in q[2:4] if s >= 0] for q in rec]
    N = numpy.zeros((S, R))
    for r in range(R):
        for s in a[r]:
            N[s, r] -= 1.0
        for s in b[r]:
            N[s, r] += 1.0

    def f(t, y):
        flux = numpy.array([kf[r] * numpy.prod(y[a[r]]) - kr[r] * numpy.prod(y[b[r]]) for r in range(R)])
        return N @ flux

    return f, numpy.array([val(c, v) for c, v in init])


def solve_ivp_values(params, x, rtol=1e-13, atol=1e-15):
    """(L*NT,) observables of the adaptive description ``params`` at point x by scipy's DOP853 at tight tolerances."""
    from scipy.integrate import solve_ivp
    par = numpy.asarray(params, dtype=numpy.float64)
    S, R, L, NT = int(par[0]), int(par[1]), int(par[2]), int(par[3])
    w = par[HDR + 8 * R + 2 * S:HDR + 8 * R + 2 * S + L * S].reshape(L, S)
    times = par[HDR + 8 * R + 2 * S + L * S:]
    f, y0 = numpy_rhs(par, x)
    sol = solve_ivp(f, (0.0, times[-1]), y0, method="DOP853", t_eval=times, rtol=rtol, atol=atol)
    assert sol.success, sol.message
    return (w @ sol.y).T.reshape(NT * L)
