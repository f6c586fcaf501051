"""Mass-action reaction network objective (VS_OBJ_MASS_ACTION, packed layout in include/varsens_b200.h).  TEST
INFRASTRUCTURE (oracle/__init__.py).

* ``values``: the C restatement (oracle/mass_action.c, frozen arithmetic shared with the device kernel) on the design points
  of oracle.cport.sample_flat -- (2+2k, rows, L) in the order fM_1, fM_2, fN_j[0..k), fN_nj[0..k).
* ``mass_action_rows`` / ``mass_action_row``: a numpy twin for use as a reference-style per-row callable (close, not
  bit-exact).
* ``chain_network`` / ``random_network``: packed descriptions used by the tests and tools/bench_mass_action.py.
"""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy

from . import cport

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def lib():
    """liboracle_ma.so, compiled on first use into the temporary directory (the source tree may be read-only), keyed by
    the source's hash; same compiler flags as oracle/Makefile."""
    global _LIB
    if _LIB is None:
        src = os.path.join(_HERE, "mass_action.c")
        tag = hashlib.sha1(open(src, "rb").read()).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "varsens_oracle_ma_%d_%s.so" % (os.getuid(), tag))
        if not os.path.exists(so):
            tmp = "%s.%d.tmp" % (so, os.getpid())
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra",
                                   "-shared", "-o", tmp, src, "-lm"])
            os.replace(tmp, so)
        L = ctypes.CDLL(so)
        L.ma_values.argtypes = [ctypes.c_int, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        _LIB = L
    return _LIB


def values(k, n, params, discard=0, scale=None, i0=0, i1=None, perm=None, raw=None):
    """(2+2k, i1-i0, L) observables of base rows [i0,i1): the arguments of oracle.cport.values."""
    i1 = n if i1 is None else i1
    par = numpy.ascontiguousarray(params, dtype=numpy.float64)
    L, rows = int(par[2]), int(i1 - i0)
    pts = numpy.concatenate([cport.sample_flat(k, n, discard, scale, t * n + i0, t * n + i1, perm, raw)
                             for t in range(2 + 2 * k)], axis=0)
    pts = numpy.ascontiguousarray(pts)
    out = numpy.empty((2 + 2 * k, rows, L))
    lib().ma_values(int(k), int(pts.shape[0]), pts.ctypes.data_as(ctypes.c_void_p), par.ctypes.data_as(ctypes.c_void_p),
                    out.ctypes.data_as(ctypes.c_void_p))
    return out


def mass_action_rows(P, params):
    """(rows, k) points -> (rows, L) observables of the packed network ``params`` (include/varsens_b200.h), classic RK4.

    numpy has no fused multiply-add and sums the stoichiometry as a matrix product, so these values are close to -- not bit
    for bit -- those of f_mass_action (oracle/mass_action.c) and the device kernel, whose arithmetic is frozen (fma, fixed order)."""
    P = numpy.atleast_2d(numpy.asarray(P, dtype=numpy.float64))
    par = numpy.asarray(params, dtype=numpy.float64)
    S, R, L, dt, nsteps = int(par[0]), int(par[1]), int(par[2]), float(par[3]), int(par[4])
    rec = par[5:5 + 8 * R].reshape(R, 8)
    init = par[5 + 8 * R:5 + 8 * R + 2 * S].reshape(S, 2)
    w = par[5 + 8 * R + 2 * S:].reshape(L, S)
    rows = P.shape[0]

    def value(coord, const):
        return P[:, int(coord)] if coord >= 0 else numpy.full(rows, const)

    kf = [value(q[4], q[5]) for q in rec]
    rev = [not (q[6] < 0 and q[7] == 0.0) for q in rec]
    kr = [value(q[6], q[7]) for q in rec]
    side = [([int(s) for s in q[0:2] if s >= 0], [int(s) for s in q[2:4] if s >= 0]) for q in rec]
    N = numpy.zeros((S, R))
    for r, (a, b) in enumerate(side):
        for s in a:
            N[s, r] -= 1.0
        for s in b:
            N[s, r] += 1.0

    def rhs(Y):
        flux = numpy.empty((rows, R))
        for r, (a, b) in enumerate(side):
            pf = numpy.prod(Y[:, a], axis=1) if a else numpy.ones(rows)
            flux[:, r] = kf[r] * pf
            if rev[r]:
                flux[:, r] -= kr[r] * (numpy.prod(Y[:, b], axis=1) if b else numpy.ones(rows))
        return flux @ N.T

    X = numpy.stack([value(c, v) for c, v in init], axis=1)
    for _ in range(nsteps):
        k1 = rhs(X)
        k2 = rhs(X + (0.5 * dt) * k1)
        k3 = rhs(X + (0.5 * dt) * k2)
        k4 = rhs(X + dt * k3)
        X = X + (dt / 6.0) * (k1 + 2.0 * k2 + 2.0 * k3 + k4)
    return X @ w.T


def mass_action_row(x, params):
    """One (k,) point -> (L,) observables: the per-row callable form (what the reference's Objective loop calls)."""
    return mass_action_rows(numpy.asarray(x)[None, :], params)[0]


def chain_network(S, dt=0.01, nsteps=1000):
    """The RK4 chain of k = 2S coordinates written as a packed mass-action network: S+1 species, S reversible reactions
    X_s <-> X_{s+1} with kf = x[s], kr = x[S+s], X(0) = e_0, one observable X_S.  Its values equal the chain's bit for bit."""
    rec = []
    for s in range(S):
        rec += [s, -1, s + 1, -1, s, 0.0, S + s, 0.0]
    init = [-1, 1.0] + [-1, 0.0] * S
    w = [0.0] * S + [1.0]
    return numpy.array([S + 1, S, 1, dt, nsteps] + rec + init + w, dtype=numpy.float64)


def random_network(seed, S, R, L, k, dt=0.01, nsteps=100):
    """A seeded packed network with reactions of order 0, 1 and 2 on either side (homodimers, catalysts, synthesis and
    degradation), reversible and irreversible reactions, and rates / initial amounts that are constants or one of the k
    coordinates.  Rates are drawn so that coordinate values in [0.5, 2] keep the dynamics tame."""
    rng = numpy.random.RandomState(seed)
    rec = []
    for r in range(R):
        order = [rng.choice(3, p=[0.15, 0.5, 0.35]) for _ in range(2)]
        side = []
        for o in order:
            sp = list(rng.randint(0, S, size=o))
            if o == 2 and rng.rand() < 0.3:
                sp[1] = sp[0]                                  # homodimer
            side.append(sp + [-1] * (2 - o))
        if S > 1 and rng.rand() < 0.15 and side[0][0] >= 0 and side[1][1] < 0:
            side[1][1] = side[0][0]                            # catalyst: on both sides
        kfc = int(rng.randint(0, k)) if rng.rand() < 0.6 else -1
        kf = 0.0 if kfc >= 0 else float(rng.uniform(0.1, 1.5))
        if rng.rand() < 0.5:
            krc, kr = -1, 0.0                                  # irreversible
        else:
            krc = int(rng.randint(0, k)) if rng.rand() < 0.5 else -1
            kr = 0.0 if krc >= 0 else float(rng.uniform(0.1, 1.5))
        rec += side[0] + side[1] + [kfc, kf, krc, kr]
    init = []
    for s in range(S):
        if rng.rand() < 0.3:
            init += [int(rng.randint(0, k)), 0.0]
        else:
            init += [-1, float(rng.uniform(0.0, 1.0))]
    w = rng.uniform(-1.0, 2.0, size=(L, S))
    w[rng.rand(L, S) < 0.5] = 0.0
    return numpy.array([S, R, L, dt, nsteps] + rec + init + list(w.ravel()), dtype=numpy.float64)
