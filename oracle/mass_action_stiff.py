"""Stiff mass-action network objective (VS_OBJ_MASS_ACTION_STIFF: an adaptive description, oracle.mass_action.adaptive_of,
integrated by Rodas3).  TEST INFRASTRUCTURE (oracle/__init__.py).

* ``points_values`` / ``values``: the C restatement (oracle/mass_action_stiff.c, frozen arithmetic shared with
  network_rosenbrock_kernel) with the signatures and results of oracle.mass_action.points_values / values_adaptive: values and
  per-trajectory {attempts, accepted, failed}, or (2+2k, rows, L*NT) values on the design points of oracle.cport.sample_flat
  and the four step counts of vs_last_network_stats.
* ``stiff_sizes``: the sizes of its sparse factor and the elimination order.

oracle/mass_action_stiff.c includes oracle/mass_action.c (one right-hand side for every network stepper) and is compiled here
into its own library, with oracle/Makefile's flags, in a temporary directory keyed by the sources' contents, so that it also
works from a read-only tree.
"""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy

from . import mass_action as ob

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = ("mass_action_stiff.c", "mass_action.c")
_CFLAGS = ["-O2", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra", "-shared"]
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        h = hashlib.sha256()
        for src in _SOURCES:
            with open(os.path.join(_HERE, src), "rb") as f:
                h.update(f.read())
        so = os.path.join(tempfile.gettempdir(), "varsens_oracle_stiff_%d_%s.so" % (os.getuid(), h.hexdigest()[:16]))
        if not os.path.exists(so):
            tmp = "%s.%d.tmp" % (so, os.getpid())
            subprocess.check_call(["gcc"] + _CFLAGS + ["-o", tmp, os.path.join(_HERE, _SOURCES[0]), "-lm"])
            os.replace(tmp, so)
        L = ctypes.CDLL(so)
        u64, i32, vp = ctypes.c_uint64, ctypes.c_int, ctypes.c_void_p
        L.ma_values_stiff.argtypes = [i32, u64, vp, vp, vp, vp]
        L.ma_stiff_sizes.argtypes = [vp, vp, vp]
        _LIB = L
    return _LIB


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def points_values(P, params):
    """(rows, k) points -> ((rows, L*NT) values, (rows, 3) int64 {attempts, accepted, failed}) of the adaptive description
    ``params`` integrated by Rodas3."""
    par = numpy.ascontiguousarray(params, dtype=numpy.float64)
    P = numpy.ascontiguousarray(numpy.atleast_2d(P), dtype=numpy.float64)
    net = ob.unpack(par, True)
    out = numpy.empty((P.shape[0], net.L * net.NT))
    info = numpy.empty((P.shape[0], 3), dtype=numpy.int64)
    lib().ma_values_stiff(int(P.shape[1]), int(P.shape[0]), _ptr(P), _ptr(par), _ptr(out), _ptr(info))
    return out, info


def values(k, n, params, discard=0, scale=None, i0=0, i1=None, perm=None, raw=None):
    """((2+2k, i1-i0, L*NT) observables, stats) of base rows [i0,i1): oracle.mass_action.values_adaptive's arguments and
    results.  stats = [accepted, rejected, failed, lane work], lane work = the sum over warps of (rows in the warp x the most
    attempts of any lane in it)."""
    out, info = points_values(ob._design(k, n, discard, scale, i0, i1, perm, raw), params)
    att = info[:, 0].reshape(2 + 2 * k, -1)
    work = 0
    for w0 in range(0, att.shape[1], ob.WARP):
        w = att[:, w0:w0 + ob.WARP]
        work += int(w.shape[1]) * int(w.max(axis=1).sum())
    acc = int(info[:, 1].sum())
    stats = numpy.array([acc, int(info[:, 0].sum()) - acc, int(info[:, 2].sum()), work], dtype=numpy.uint64)
    return out.reshape(2 + 2 * k, att.shape[1], -1), stats


def stiff_sizes(params):
    """The Rodas3 factor of the adaptive description ``params``: dict(nlu = nonzeros of L+U with the diagonal, nlow / nup =
    entries below / above the diagonal, nupd = update operations of one factorisation, ncol = Jacobian columns (reaction,
    species), njt = Jacobian scatter targets, ord = the elimination order)."""
    par = numpy.ascontiguousarray(params, dtype=numpy.float64)
    net = ob.unpack(par, True)
    sizes = numpy.zeros(6, dtype=numpy.int64)
    ord_ = numpy.zeros(net.S, dtype=numpy.int64)
    lib().ma_stiff_sizes(_ptr(par), _ptr(sizes), _ptr(ord_))
    return dict(zip(("nlu", "nlow", "nup", "nupd", "ncol", "njt"), (int(v) for v in sizes)), ord=ord_)
