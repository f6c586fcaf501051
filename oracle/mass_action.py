"""Mass-action reaction network objectives (VS_OBJ_MASS_ACTION, VS_OBJ_MASS_ACTION_ADAPTIVE, packed layouts in
include/varsens_b200.h).  TEST INFRASTRUCTURE (oracle/__init__.py).

* ``unpack`` / ``pack``: the one reader and writer of the packed layouts here.  A network is edited (truncated, a reaction
  appended) by unpacking it, changing the fields and packing it again.
* ``values`` / ``values_adaptive`` / ``points_values``: the C restatement (oracle/mass_action.c, frozen arithmetic shared
  with the device kernels) on the design points of oracle.cport.sample_flat -- (2+2k, rows, L) or (2+2k, rows, L*NT) in the
  order fM_1, fM_2, fN_j[0..k), fN_nj[0..k); the adaptive form also returns the four step counts of vs_last_network_stats.
* ``mass_action_rows`` / ``mass_action_row``: a numpy twin of the fixed step for use as a reference-style per-row callable
  (close, not bit-exact).  ``numpy_rhs`` / ``solve_ivp_values``: a numpy right-hand side and a tight
  scipy.integrate.solve_ivp reference for the adaptive description.
* ``chain_network`` / ``random_network``: packed fixed-step descriptions used by the tests and tools; ``adaptive_of`` turns
  one into an adaptive description.
"""
import ctypes
import dataclasses

import numpy

from . import cport

WARP = 32          # the adaptive kernel's warps: 32 consecutive rows of one design point
# the header scalars after S R L (fixed step) and after S R L NT (adaptive)
HEAD = {False: ("dt", "nsteps"), True: ("rtol", "atol", "h0", "max_steps")}


@dataclasses.dataclass
class Network:
    """The fields of a packed description.  S, R, L, NT and the kernels' table sizes nnz / nobs follow from the arrays."""
    rec: numpy.ndarray            # (R, 8): reactant, reactant, product, product (-1: none), kf coord, kf, kr coord, kr
    init: numpy.ndarray           # (S, 2): coordinate (-1: none), constant
    w: numpy.ndarray              # (L, S) observable weights
    head: dict                    # the scalars named by HEAD
    times: numpy.ndarray = None   # (NT,) output times; None for the fixed step

    S = property(lambda self: len(self.init))
    R = property(lambda self: len(self.rec))
    L = property(lambda self: len(self.w))
    NT = property(lambda self: len(self.times))
    nobs = property(lambda self: int(numpy.count_nonzero(self.w)), doc="Nonzero weights: the observable lists' entries.")
    nnz = property(lambda self: int(numpy.count_nonzero(self.N)),
                   doc="Nonzero net coefficients: the entries of the species-major stoichiometry list.")

    @property
    def N(self):
        """(S, R) net stoichiometric coefficients, products - reactants."""
        N = numpy.zeros((self.S, self.R))
        for r, q in enumerate(self.rec):
            for j, s in enumerate(q[:4]):
                if s >= 0:
                    N[int(s), r] += 1.0 if j >= 2 else -1.0
        return N


def unpack(params, adaptive):
    """The Network of the packed description ``params``, fixed-step or adaptive; its arrays are views of a copy."""
    par = numpy.array(params, dtype=numpy.float64)
    S, R, L = (int(v) for v in par[:3])
    o = 3 + int(adaptive)
    head = dict(zip(HEAD[adaptive], par[o:]))
    ends = numpy.cumsum([o + len(HEAD[adaptive]), 8 * R, 2 * S, L * S, int(par[3]) if adaptive else 0])
    assert ends[-1] == par.size, "%d values are not a packed %s network" % (par.size, "adaptive" if adaptive else "fixed-step")
    rec, init, w, times = (par[a:b] for a, b in zip(ends[:-1], ends[1:]))
    return Network(rec.reshape(R, 8), init.reshape(S, 2), w.reshape(L, S), head, times if adaptive else None)


def pack(net):
    """The packed description of the Network ``net``: the inverse of unpack."""
    adaptive = net.times is not None
    head = [net.S, net.R, net.L] + ([net.NT] if adaptive else []) + [net.head[h] for h in HEAD[adaptive]]
    return numpy.concatenate([numpy.asarray(a, dtype=numpy.float64).ravel()
                              for a in [head, net.rec, net.init, net.w] + ([net.times] if adaptive else [])])


def _design(k, n, discard, scale, i0, i1, perm, raw):
    """The points of base rows [i0,i1) of every block in turn (the arguments of oracle.cport.values)."""
    i1 = n if i1 is None else i1
    return numpy.concatenate([cport.sample_flat(k, n, discard, scale, t * n + i0, t * n + i1, perm, raw)
                              for t in range(2 + 2 * k)], axis=0)


def values(k, n, params, discard=0, scale=None, i0=0, i1=None, perm=None, raw=None):
    """(2+2k, i1-i0, L) observables of base rows [i0,i1): the arguments of oracle.cport.values."""
    pts = _design(k, n, discard, scale, i0, i1, perm, raw)
    par = numpy.ascontiguousarray(params, dtype=numpy.float64)
    L = unpack(par, False).L
    out = numpy.empty((pts.shape[0], L))
    cport.lib().ma_values(int(k), int(pts.shape[0]), pts.ctypes.data_as(ctypes.c_void_p), par.ctypes.data_as(ctypes.c_void_p),
                          out.ctypes.data_as(ctypes.c_void_p))
    return out.reshape(2 + 2 * k, -1, L)


def points_values(P, params):
    """(rows, k) points -> ((rows, L*NT) values, (rows, 3) int64 {attempts, accepted, failed}) of the adaptive ``params``."""
    par = numpy.ascontiguousarray(params, dtype=numpy.float64)
    P = numpy.ascontiguousarray(numpy.atleast_2d(P), dtype=numpy.float64)
    net = unpack(par, True)
    out = numpy.empty((P.shape[0], net.L * net.NT))
    info = numpy.empty((P.shape[0], 3), dtype=numpy.int64)
    cport.lib().ma_values_adaptive(int(P.shape[1]), int(P.shape[0]), P.ctypes.data_as(ctypes.c_void_p),
                                   par.ctypes.data_as(ctypes.c_void_p), out.ctypes.data_as(ctypes.c_void_p),
                                   info.ctypes.data_as(ctypes.c_void_p))
    return out, info


def values_adaptive(k, n, params, discard=0, scale=None, i0=0, i1=None, perm=None, raw=None):
    """((2+2k, i1-i0, L*NT) observables, stats) of base rows [i0,i1): the arguments of values.  stats = [accepted, rejected,
    failed, lane work] over these rows, lane work = the sum over warps of (rows in the warp x the most attempts of any lane
    in it)."""
    out, info = points_values(_design(k, n, discard, scale, i0, i1, perm, raw), params)
    att = info[:, 0].reshape(2 + 2 * k, -1)
    work = 0
    for w0 in range(0, att.shape[1], WARP):
        w = att[:, w0:w0 + WARP]
        work += int(w.shape[1]) * int(w.max(axis=1).sum())
    acc = int(info[:, 1].sum())
    stats = numpy.array([acc, int(info[:, 0].sum()) - acc, int(info[:, 2].sum()), work], dtype=numpy.uint64)
    return out.reshape(2 + 2 * k, att.shape[1], -1), stats


def mass_action_rows(P, params):
    """(rows, k) points -> (rows, L) observables of the packed fixed-step network ``params``, classic RK4.

    numpy has no fused multiply-add and sums the stoichiometry as a matrix product, so these values are close to -- not bit
    for bit -- those of f_mass_action (oracle/mass_action.c) and the device kernel, whose arithmetic is frozen (fma, fixed order)."""
    P = numpy.atleast_2d(numpy.asarray(P, dtype=numpy.float64))
    net = unpack(params, False)
    dt, N, rows = float(net.head["dt"]), net.N, P.shape[0]

    def value(coord, const):
        return P[:, int(coord)] if coord >= 0 else numpy.full(rows, const)

    kf = [value(q[4], q[5]) for q in net.rec]
    rev = [not (q[6] < 0 and q[7] == 0.0) for q in net.rec]
    kr = [value(q[6], q[7]) for q in net.rec]
    side = [([int(s) for s in q[0:2] if s >= 0], [int(s) for s in q[2:4] if s >= 0]) for q in net.rec]

    def rhs(Y):
        flux = numpy.empty((rows, net.R))
        for r, (a, b) in enumerate(side):
            pf = numpy.prod(Y[:, a], axis=1) if a else numpy.ones(rows)
            flux[:, r] = kf[r] * pf
            if rev[r]:
                flux[:, r] -= kr[r] * (numpy.prod(Y[:, b], axis=1) if b else numpy.ones(rows))
        return flux @ N.T

    X = numpy.stack([value(c, v) for c, v in net.init], axis=1)
    for _ in range(int(net.head["nsteps"])):
        k1 = rhs(X)
        k2 = rhs(X + (0.5 * dt) * k1)
        k3 = rhs(X + (0.5 * dt) * k2)
        k4 = rhs(X + dt * k3)
        X = X + (dt / 6.0) * (k1 + 2.0 * k2 + 2.0 * k3 + k4)
    return X @ net.w.T


def mass_action_row(x, params):
    """One (k,) point -> (L,) observables: the per-row callable form (what the reference's Objective loop calls)."""
    return mass_action_rows(numpy.asarray(x)[None, :], params)[0]


def numpy_rhs(params, x):
    """f(t, y) of the adaptive description ``params`` at the scaled point x, for solve_ivp, and y(0)."""
    net = unpack(params, True)
    x = numpy.asarray(x, dtype=numpy.float64)
    val = lambda c, v: x[int(c)] if c >= 0 else v                   # noqa: E731
    kf = numpy.array([val(q[4], q[5]) for q in net.rec])
    kr = numpy.array([val(q[6], q[7]) for q in net.rec])
    a = [[int(s) for s in q[0:2] if s >= 0] for q in net.rec]
    b = [[int(s) for s in q[2:4] if s >= 0] for q in net.rec]
    N, R = net.N, net.R

    def f(t, y):
        flux = numpy.array([kf[r] * numpy.prod(y[a[r]]) - kr[r] * numpy.prod(y[b[r]]) for r in range(R)])
        return N @ flux

    return f, numpy.array([val(c, v) for c, v in net.init])


def solve_ivp_values(params, x, rtol=1e-13, atol=1e-15):
    """(L*NT,) observables of the adaptive description ``params`` at point x by scipy's DOP853 at tight tolerances."""
    from scipy.integrate import solve_ivp
    net = unpack(params, True)
    f, y0 = numpy_rhs(params, x)
    sol = solve_ivp(f, (0.0, net.times[-1]), y0, method="DOP853", t_eval=net.times, rtol=rtol, atol=atol)
    assert sol.success, sol.message
    return (net.w @ sol.y).T.reshape(net.NT * net.L)


def adaptive_of(packed, times, rtol=1e-6, atol=1e-9, h0=None, max_steps=100000):
    """The fixed-step description ``packed`` as an adaptive one with output times ``times``; h0 = None is 1e-6 * times[-1],
    as in AdaptiveMassActionNetwork."""
    net = unpack(packed, False)
    net.times = numpy.atleast_1d(numpy.asarray(times, dtype=numpy.float64))
    h0 = 1e-6 * float(net.times[-1]) if h0 is None else float(h0)
    net.head = dict(rtol=float(rtol), atol=float(atol), h0=h0, max_steps=float(max_steps))
    return pack(net)


def chain_network(S, dt=0.01, nsteps=1000):
    """The RK4 chain of k = 2S coordinates written as a packed mass-action network: S+1 species, S reversible reactions
    X_s <-> X_{s+1} with kf = x[s], kr = x[S+s], X(0) = e_0, one observable X_S.  Its values equal the chain's bit for bit."""
    rec = [[s, -1, s + 1, -1, s, 0.0, S + s, 0.0] for s in range(S)]
    init = [[-1, 1.0]] + [[-1, 0.0]] * S
    return pack(Network(rec, init, [[0.0] * S + [1.0]], dict(dt=dt, nsteps=nsteps)))


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
        rec.append(side[0] + side[1] + [kfc, kf, krc, kr])
    init = []
    for s in range(S):
        if rng.rand() < 0.3:
            init.append([int(rng.randint(0, k)), 0.0])
        else:
            init.append([-1, float(rng.uniform(0.0, 1.0))])
    w = rng.uniform(-1.0, 2.0, size=(L, S))
    w[rng.rand(L, S) < 0.5] = 0.0
    return pack(Network(rec, init, w, dict(dt=dt, nsteps=nsteps)))
