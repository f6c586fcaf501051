"""ctypes front end of liboracle.so (oracle/oracle.c; oracle/mass_action.c's entry points are called from
oracle/mass_action.py).  TEST INFRASTRUCTURE (oracle/__init__.py)."""
import ctypes
import os
import subprocess

import numpy

from . import pipeline as _pipeline

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

OBJ_GFUNCTION, OBJ_ISHIGAMI, OBJ_RK4_CHAIN = 0, 1, 2
SCALE_IDENTITY, SCALE_LINEAR, SCALE_POWER = 0, 1, 2


def build(force=False):
    so = os.path.join(_HERE, "liboracle.so")
    newest = max(os.path.getmtime(os.path.join(_HERE, src)) for src in ("oracle.c", "mass_action.c"))
    if force or not os.path.exists(so) or os.path.getmtime(so) < newest:
        subprocess.check_call(["make", "-s", "-C", _HERE, "liboracle.so"])
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = ctypes.CDLL(build())
        u64, i32, vp = ctypes.c_uint64, ctypes.c_int, ctypes.c_void_p
        L.orc_num_threads.restype = i32
        L.orc_set_threads.argtypes = [i32]
        L.orc_halton.argtypes = [i32, u64, u64, vp]
        L.orc_sample_flat.argtypes = [i32, u64, u64, vp, vp, i32, vp, vp, u64, u64, vp]
        L.orc_values.argtypes = [i32, u64, u64, vp, vp, i32, vp, vp, i32, vp, u64, u64, vp]
        L.orc_sums.argtypes = [i32, u64, u64, vp, vp, i32, vp, vp, i32, vp, u64, u64, i32, vp, vp]
        L.ma_values.argtypes = [i32, u64, vp, vp, vp]
        L.ma_values_adaptive.argtypes = [i32, u64, vp, vp, vp, vp]
        _LIB = L
    return _LIB


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _scale_args(k, scale):
    """scale = None | ('linear', lb, ub) | ('power', lb, ub) -> (kind, lb, w_or_r) as varsens/scale.py:33,62."""
    if scale is None:
        return SCALE_IDENTITY, None, None
    kind, lb, ub = scale
    lb = numpy.ascontiguousarray(numpy.broadcast_to(numpy.asarray(lb, dtype=numpy.float64), (k,)))
    ub = numpy.ascontiguousarray(numpy.broadcast_to(numpy.asarray(ub, dtype=numpy.float64), (k,)))
    if kind == 'linear':
        return SCALE_LINEAR, lb, numpy.ascontiguousarray(ub - lb)
    return SCALE_POWER, lb, numpy.ascontiguousarray(ub / lb)


def _perm32(n, perm):
    perm = _pipeline.permutation(n) if perm is None else perm
    return numpy.ascontiguousarray(perm, dtype=numpy.uint32)


def halton(k, first_index, count):
    out = numpy.empty((int(count), int(k)))
    lib().orc_halton(int(k), int(first_index), int(count), _ptr(out))
    return out


def sample_flat(k, n, discard=0, scale=None, row_begin=0, row_end=None, perm=None, raw=None):
    row_end = 2 * n * (1 + k) if row_end is None else row_end
    kind, lb, wr = _scale_args(k, scale)
    perm = _perm32(n, perm)
    raw = None if raw is None else numpy.ascontiguousarray(raw, dtype=numpy.float64)
    out = numpy.empty((int(row_end - row_begin), int(k)))
    lib().orc_sample_flat(int(k), int(n), int(discard), _ptr(perm), _ptr(raw), kind, _ptr(lb), _ptr(wr),
                          int(row_begin), int(row_end), _ptr(out))
    return out


def values(k, n, objective, params, discard=0, scale=None, i0=0, i1=None, perm=None, raw=None):
    """(2+2k, i1-i0) objective values: rows fM_1, fM_2, fN_j[0..k), fN_nj[0..k)."""
    i1 = n if i1 is None else i1
    kind, lb, wr = _scale_args(k, scale)
    perm = _perm32(n, perm)
    raw = None if raw is None else numpy.ascontiguousarray(raw, dtype=numpy.float64)
    par = numpy.ascontiguousarray(params, dtype=numpy.float64)
    out = numpy.empty((2 + 2 * k, int(i1 - i0)))
    lib().orc_values(int(k), int(n), int(discard), _ptr(perm), _ptr(raw), kind, _ptr(lb), _ptr(wr),
                     int(objective), _ptr(par), int(i0), int(i1), _ptr(out))
    return out


def sums(k, n, objective, params, discard=0, scale=None, i0=0, i1=None, perm=None, raw=None, second_order=True):
    """Long-double sufficient statistics of base rows [i0,i1) as oracle.pipeline's sums dict."""
    i1 = n if i1 is None else i1
    kind, lb, wr = _scale_args(k, scale)
    perm = _perm32(n, perm)
    raw = None if raw is None else numpy.ascontiguousarray(raw, dtype=numpy.float64)
    par = numpy.ascontiguousarray(params, dtype=numpy.float64)
    m = 2 + 2 * k
    s = numpy.zeros(m, dtype=numpy.longdouble)
    g = numpy.zeros((m, m), dtype=numpy.longdouble)
    lib().orc_sums(int(k), int(n), int(discard), _ptr(perm), _ptr(raw), kind, _ptr(lb), _ptr(wr),
                   int(objective), _ptr(par), int(i0), int(i1), int(bool(second_order)), _ptr(s), _ptr(g))
    J, N = slice(2, 2 + k), slice(2 + k, m)
    return dict(s_ab=g[0, 1], s_a=s[0], s_b=s[1], q_a=g[0, 0], q_b=g[1, 1],
                aJ=g[0, J], bN=g[1, N], aN=g[0, N], bJ=g[1, J],
                NJ=g[N, J].copy(), NN=g[N, N].copy(), JJ=g[J, J].copy())


def run(k, n, objective, params, discard=0, scale=None, perm=None, raw=None, second_order=True):
    """Indices dict (oracle.pipeline.indices_from_sums) for the whole design."""
    return _pipeline.indices_from_sums(
        sums(k, n, objective, params, discard, scale, 0, n, perm, raw, second_order), k, n)
