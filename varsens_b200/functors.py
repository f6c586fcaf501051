"""Registered device objective functors.

The reference calls a Python callable once per sample row (varsens/saltelli.py:308-353).  An
instance of one of these classes can be passed wherever the reference takes ``objective_func`` /
``objective``; the evaluation then happens inside the CUDA kernels (fused with generation and
the estimator reductions when a fused kernel exists for k, otherwise through the two-phase
eval-to-HBM + Gram path).  They carry no host implementation: there is no CPU fallback.
"""
import warnings

import numpy

from . import _cabi


class Functor(object):
    objective_id = None
    separable = False

    def params(self, k):
        raise NotImplementedError

    def outputs(self, k):
        """Outputs per sample point (the l of fM_1 (n, l) and sens (k, l))."""
        return 1

    def check_run(self, ctx):
        """Called after ctx evaluated this functor (Objective values, or a Varsens step on this process's rows)."""

    def __call__(self, x):
        raise _cabi.VarsensError(
            "%s is a device functor: pass it to Objective/Varsens instead of calling it on the host"
            % type(self).__name__)


class GFunction(Functor):
    """Sobol g-function  prod_c (|4 x_c - 2| + a_c) / (1 + a_c)
    (varsens/tests/test_g_function.py:9-13, README.md:33-36)."""
    objective_id = _cabi.OBJ_GFUNCTION
    separable = True

    def __init__(self, a):
        self.a = numpy.asarray(a, dtype=numpy.float64).copy()

    def params(self, k):
        if self.a.shape != (k,):
            raise _cabi.VarsensError("GFunction has %d coefficients, k = %d" % (self.a.size, k))
        return self.a


class Ishigami(Functor):
    """sin x0 + A sin^2 x1 + B x2^4 sin x0  (BASELINE.json config 2)."""
    objective_id = _cabi.OBJ_ISHIGAMI

    def __init__(self, A=7.0, B=0.1):
        self.A, self.B = float(A), float(B)

    def params(self, k):
        return numpy.array([self.A, self.B])


class RK4Chain(Functor):
    """Fixed-step RK4 of the reversible mass-action chain X_0 <-> ... <-> X_{k/2}; the k parameters are the
    forward (first half) and reverse (second half) rate constants; objective = X_{k/2}(nsteps*dt)
    (BASELINE.json config 5; spec frozen in include/varsens_b200.h)."""
    objective_id = _cabi.OBJ_RK4_CHAIN

    def __init__(self, dt=0.01, nsteps=1000):
        self.dt, self.nsteps = float(dt), int(nsteps)

    def params(self, k):
        return numpy.array([self.dt, float(self.nsteps)])


class Param(object):
    """Coordinate ``c`` of the (scaled) sample point, as a rate constant or initial amount of a MassActionNetwork."""

    def __init__(self, c):
        if isinstance(c, bool) or not isinstance(c, (int, numpy.integer)) or c < 0:
            raise _cabi.VarsensError("Param needs a coordinate index >= 0, got %r" % (c,))
        self.c = int(c)

    def __repr__(self):
        return "Param(%d)" % self.c


class _Network(Functor):
    """The parsing MassActionNetwork and AdaptiveMassActionNetwork share: species, reactions, initial amounts and observables
    as the packed records, initial amounts and weights of include/varsens_b200.h (``self._body``)."""

    def __init__(self, species, reactions, initial, observables):
        err = _cabi.VarsensError
        what = type(self).__name__
        if isinstance(species, (int, numpy.integer)) and not isinstance(species, bool):
            self.names = None
            S = int(species)
        else:
            self.names = [str(s) for s in species]
            if len(set(self.names)) != len(self.names):
                raise err("%s: species names are not unique" % what)
            S = len(self.names)
        if not 1 <= S <= 128:
            raise err("%s: %d species, need 1..128" % (what, S))
        self.S = S
        self._max_coord = -1                       # largest sample coordinate a Param refers to
        reactions = list(reactions)
        if not 1 <= len(reactions) <= 512:
            raise err("%s: %d reactions, need 1..512" % (what, len(reactions)))
        recs = []
        for r, rx in enumerate(reactions):
            rx = tuple(rx)
            if len(rx) not in (3, 4):
                raise err("%s: reaction %d must be (reactants, products, kf[, kr])" % (what, r))
            a = self._side(rx[0], "reaction %d reactants" % r)
            b = self._side(rx[1], "reaction %d products" % r)
            kfc, kf = self._value(rx[2], "reaction %d kf" % r)
            kr = rx[3] if len(rx) == 4 else None
            krc, krv = (-1, 0.0) if kr is None else self._value(kr, "reaction %d kr" % r)
            recs.append(a + b + [kfc, kf, krc, krv])
        initial = list(initial)
        if len(initial) != S:
            raise err("%s: %d initial amounts for %d species" % (what, len(initial), S))
        init = [self._value(v, "initial amount of species %d" % s) for s, v in enumerate(initial)]
        observables = list(observables)
        if not 1 <= len(observables) <= 64:
            raise err("%s: %d observables, need 1..64" % (what, len(observables)))
        w = numpy.zeros((len(observables), S))
        for o, ob in enumerate(observables):
            items = ob.items() if isinstance(ob, dict) else [(ob, 1.0)]
            for sp, wt in items:
                if isinstance(wt, Param) or isinstance(wt, bool) or not isinstance(wt, (int, float, numpy.number)):
                    raise err("%s: observable %d, weight %r is not a number" % (what, o, wt))
                w[o, self._species(sp, "observable %d" % o)] += float(wt)
        self.L = len(observables)
        self.R = len(recs)
        self._body = [x for rec in recs for x in rec] + [x for iv in init for x in iv] + list(w.ravel())

    def _species(self, sp, what):
        err = _cabi.VarsensError
        if isinstance(sp, str):
            if self.names is None or sp not in self.names:
                raise err("%s: %s: unknown species %r" % (type(self).__name__, what, sp))
            return self.names.index(sp)
        if isinstance(sp, bool) or not isinstance(sp, (int, numpy.integer)) or not 0 <= sp < self.S:
            raise err("%s: %s: species %r is neither a name nor an index in [0, %d)" % (type(self).__name__, what, sp, self.S))
        return int(sp)

    def _side(self, side, what):
        if side is None:
            side = []
        elif isinstance(side, (str, int, numpy.integer)):
            side = [side]
        side = [self._species(sp, what) for sp in side]
        if len(side) > 2:
            raise _cabi.VarsensError("%s: %s: %d species, at most 2" % (type(self).__name__, what, len(side)))
        return side + [-1] * (2 - len(side))

    def _value(self, v, what):
        if isinstance(v, Param):
            self._max_coord = max(self._max_coord, v.c)
            return [v.c, 0.0]
        if isinstance(v, bool) or not isinstance(v, (int, float, numpy.number)):
            raise _cabi.VarsensError("%s: %s = %r: need a number or Param(c)" % (type(self).__name__, what, v))
        return [-1, float(v)]

    def params(self, k):
        if self._max_coord >= k:
            raise _cabi.VarsensError("%s uses coordinate %d, the sample has k = %d" % (type(self).__name__, self._max_coord, k))
        _cabi.objective_outputs(k, self.objective_id, self._packed)          # the library's own validation
        return self._packed

    def outputs(self, k):
        return _cabi.objective_outputs(k, self.objective_id, self.params(k))


class MassActionNetwork(_Network):
    """Mass-action reaction network integrated by classic fixed-step RK4 on the GPU; the objective is L observables, each a
    weighted sum of species amounts at T = nsteps * dt (the l = L outputs of every sample point).

    ``species``      a count, or a list of names;
    ``reactions``    tuples ``(reactants, products, kf, kr=None)``: each side a species, a list of at most two species (a
                     species may appear twice) or an empty list; species by name or index; ``kr=None`` = irreversible;
    ``initial``      one initial amount per species;
    ``observables``  a list of ``{species: weight}`` dicts or of single species (weight 1).
    A rate or initial amount is a number (a constant) or ``Param(c)``: coordinate c of the scaled sample point.  Packed
    layout and frozen arithmetic: include/varsens_b200.h (VS_OBJ_MASS_ACTION)."""
    objective_id = _cabi.OBJ_MASS_ACTION

    def __init__(self, species, reactions, initial, observables, dt=0.01, nsteps=1000):
        err = _cabi.VarsensError
        self.dt = float(dt)
        if not numpy.isfinite(self.dt):
            raise err("MassActionNetwork: dt = %r is not finite" % (dt,))
        if isinstance(nsteps, bool) or not isinstance(nsteps, (int, numpy.integer)) or not 0 <= nsteps < 2 ** 31:
            raise err("MassActionNetwork: nsteps = %r, need an integer in [0, 2^31)" % (nsteps,))
        self.nsteps = int(nsteps)
        _Network.__init__(self, species, reactions, initial, observables)
        self._packed = numpy.array([self.S, self.R, self.L, self.dt, self.nsteps] + self._body, dtype=numpy.float64)


class AdaptiveMassActionNetwork(_Network):
    """Mass-action reaction network integrated by adaptive Dormand-Prince 5(4) on the GPU: every trajectory picks its own
    steps to meet ``rtol`` / ``atol`` and lands exactly on each of the output ``times`` (0 < t_1 < ... < t_NT; integration
    starts at t = 0).  The objective has l = L * NT outputs per sample point, column m*L + o = observable o at time t_{m+1},
    so ``Objective.fM_1.reshape(n, NT, L)`` is the time course.

    ``species``, ``reactions``, ``initial`` and ``observables`` are those of MassActionNetwork; L * NT <= 64.
    ``rtol`` >= 0, ``atol`` > 0: the error of a step is measured against rtol * |X_s| + atol per species;
    ``h0``           the first step (None: 1e-6 * times[-1]);
    ``max_steps``    attempted steps per trajectory before it is marked failed;
    ``method``       "dopri5" (explicit, VS_OBJ_MASS_ACTION_ADAPTIVE) or "rodas3": the L-stable Rosenbrock method for stiff
                     networks, whose rates lie orders of magnitude apart (VS_OBJ_MASS_ACTION_STIFF; same packed parameters).
    A failed trajectory (more than max_steps attempts, or a step too small to advance t) gives NaN from the output time it
    could not reach on; Objective and Varsens then issue a RuntimeWarning with the count.  Packed layout and frozen arithmetic:
    include/varsens_b200.h (VS_OBJ_MASS_ACTION_ADAPTIVE, VS_OBJ_MASS_ACTION_STIFF)."""
    objective_id = _cabi.OBJ_MASS_ACTION_ADAPTIVE                       # of the default method; each instance sets its own
    METHODS = {"dopri5": _cabi.OBJ_MASS_ACTION_ADAPTIVE, "rodas3": _cabi.OBJ_MASS_ACTION_STIFF}

    def __init__(self, species, reactions, initial, observables, times, rtol=1e-6, atol=1e-9, h0=None, max_steps=100000,
                 method="dopri5"):
        err = _cabi.VarsensError
        if not isinstance(method, str) or method not in self.METHODS:
            raise err("AdaptiveMassActionNetwork: method = %r, need one of %s" % (method, sorted(self.METHODS)))
        self.method, self.objective_id = method, self.METHODS[method]
        _Network.__init__(self, species, reactions, initial, observables)
        try:
            t = numpy.asarray(times, dtype=numpy.float64)
        except (TypeError, ValueError):
            raise err("AdaptiveMassActionNetwork: times = %r is not a list of numbers" % (times,))
        if t.ndim != 1 or t.size < 1 or not numpy.isfinite(t).all() or t[0] <= 0 or (numpy.diff(t) <= 0).any():
            raise err("AdaptiveMassActionNetwork: times must be finite and 0 < t_1 < t_2 < ..., got %r" % (times,))
        if self.L * t.size > 64:
            raise err("AdaptiveMassActionNetwork: %d observables at %d times are %d outputs, at most 64" % (self.L, t.size,
                                                                                                           self.L * t.size))
        h0 = 1e-6 * float(t[-1]) if h0 is None else h0
        for name, v, lo_ok in (("rtol", rtol, lambda v: v >= 0), ("atol", atol, lambda v: v > 0), ("h0", h0, lambda v: v > 0)):
            if isinstance(v, bool) or not isinstance(v, (int, float, numpy.number)) or not numpy.isfinite(v) or not lo_ok(v):
                raise err("AdaptiveMassActionNetwork: %s = %r is out of range" % (name, v))
        if isinstance(max_steps, bool) or not isinstance(max_steps, (int, numpy.integer)) or not 1 <= max_steps < 2 ** 31:
            raise err("AdaptiveMassActionNetwork: max_steps = %r, need an integer in [1, 2^31)" % (max_steps,))
        self.times, self.rtol, self.atol, self.h0, self.max_steps = t.copy(), float(rtol), float(atol), float(h0), int(max_steps)
        self._packed = numpy.array([self.S, self.R, self.L, t.size, self.rtol, self.atol, self.h0, self.max_steps] + self._body +
                                   list(t), dtype=numpy.float64)

    def check_run(self, ctx):
        failed = ctx.network_stats()["failed"]
        if failed:
            warnings.warn("AdaptiveMassActionNetwork: %d trajectories failed (more than max_steps = %d attempts, or a step too "
                          "small to advance t); their outputs from the failing time on are NaN" % (failed, self.max_steps),
                          RuntimeWarning, stacklevel=3)


def vectorized(fn):
    """Mark a Python objective as vectorised: it receives a (rows, k) CUDA torch.float64 tensor of
    sample rows and returns a (rows,) or (rows, l) tensor.  Sample rows are materialised on the GPU
    in batches (export-mode kernel) and never leave it; only the callable itself is user code."""
    fn.varsens_vectorized = True
    return fn
