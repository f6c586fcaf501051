"""ctypes binding of libvarsens_b200.so (include/varsens_b200.h).

The library is the only compute path: if it is missing or no CUDA device is present the calls
raise -- there is no CPU fallback (BASELINE.json north_star).
"""
import ctypes
import os
import threading

import numpy

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VS_LIB") or os.path.join(_HERE, "libvarsens_b200.so")   # VS_LIB: alternative builds (kernel experiments)

VS_OK = 0
MEM_HOST, MEM_DEVICE = 0, 1
SCALE_IDENTITY, SCALE_LINEAR, SCALE_POWER = 0, 1, 2
OBJ_GFUNCTION, OBJ_ISHIGAMI, OBJ_RK4_CHAIN, OBJ_MASS_ACTION, OBJ_MASS_ACTION_ADAPTIVE, OBJ_MASS_ACTION_STIFF = 0, 1, 2, 3, 4, 5
NETWORK_STATS = ("accepted", "rejected", "failed", "lane_work")      # vs_last_network_stats, in order
FLAG_SECOND_ORDER, FLAG_SEPARABLE = 1, 2

# every symbol include/varsens_b200.h declares (tests/test_cabi_symbols.py checks the header against this)
SYMBOLS = (
    "vs_abi_version", "vs_last_error", "vs_ctx_create", "vs_ctx_destroy", "vs_ctx_set_stream",
    "vs_ctx_synchronize", "vs_ctx_launch_count", "vs_halton_bases", "vs_halton_terms", "vs_partials_len",
    "vs_halton", "vs_sobol", "vs_sample_flat", "vs_eval_values", "vs_partials_from_values", "vs_finalize",
    "vs_finalize_device", "vs_allreduce_finalize_p2p", "vs_indices_from_values", "vs_fused_partials", "vs_run_fused", "vs_measure_fp64_peak", "vs_last_kernel_ms",
    "vs_ctx_reload_env", "vs_ctx_set_halton_mode", "vs_halton_terms_mode", "vs_run_fused_p2p", "vs_last_tail_ns",
    "vs_halton_arith_check", "vs_reference_permutation", "vs_ctx_set_timing", "vs_sample_flat_shard",
    "vs_objective_outputs", "vs_last_network_stats",
)
HALTON_DIVIDE, HALTON_RECIPROCAL, HALTON_RUNNING_RECIPROCAL, HALTON_HORNER = 0, 1, 2, 3
ERR_TIMEOUT = 6


class VarsensError(RuntimeError):
    status = None


class vs_scale(ctypes.Structure):
    _fields_ = [("kind", ctypes.c_int), ("lower", ctypes.c_void_p), ("upper", ctypes.c_void_p)]


def _result_fields(k, l, second_order=True):
    """(name, length, shape) of each array of a result block, in the library's order; a first-order block ends after sens_t."""
    kl = k * l
    fields = [("E_2", l, (l,)), ("var_y", l, (l,)), ("U_j", kl, (k, l)), ("U_nj", kl, (k, l)), ("sens", kl, (k, l)),
              ("sens_t", kl, (k, l)), ("sens_2", kl * kl, (k, l, k, l)), ("sens_2n", kl * kl, (k, l, k, l))]
    return fields if second_order else fields[:6]


def _block_len(k, l, second_order=True):
    return sum(cnt for _, cnt, _ in _result_fields(k, l, second_order))


class vs_result(ctypes.Structure):
    _fields_ = [(name, ctypes.c_void_p) for name, _, _ in _result_fields(1, 1)]


_lib = None
_lock = threading.Lock()


def lib():
    """Load the shared library (once).  Raises VarsensError if it has not been built."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise VarsensError(
                "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(make -C varsens_b200/csrc).  varsens_b200 has no CPU fallback." % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        u64, i32, vp, sz = ctypes.c_uint64, ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t
        P = ctypes.POINTER
        L.vs_abi_version.restype = i32
        L.vs_last_error.restype = ctypes.c_char_p
        L.vs_ctx_create.argtypes = [i32, P(vp)]
        L.vs_ctx_destroy.argtypes = [vp]
        L.vs_ctx_set_stream.argtypes = [vp, vp]
        L.vs_ctx_synchronize.argtypes = [vp]
        L.vs_ctx_launch_count.argtypes = [vp]
        L.vs_ctx_launch_count.restype = u64
        L.vs_halton_bases.argtypes = [i32, vp]
        L.vs_halton_terms.argtypes = [i32, u64, vp, vp, vp, u64, P(u64)]
        L.vs_partials_len.argtypes = [i32, i32]
        L.vs_partials_len.restype = sz
        L.vs_halton.argtypes = [vp, i32, u64, u64, P(vs_scale), vp, i32]
        L.vs_sobol.argtypes = [vp, i32, u64, u64, vp, i32, P(vs_scale), vp, i32]
        L.vs_sample_flat.argtypes = [vp, i32, u64, u64, vp, i32, vp, i32, P(vs_scale), u64, u64, vp, i32]
        L.vs_eval_values.argtypes = [vp, i32, u64, u64, vp, i32, vp, i32, P(vs_scale), i32, vp, i32, u64, u64, vp, i32]
        L.vs_partials_from_values.argtypes = [vp, i32, i32, u64, vp, i32, vp, i32, vp, i32]
        L.vs_finalize.argtypes = [vp, i32, i32, u64, u64, vp, i32, i32, P(vs_result)]
        L.vs_finalize_device.argtypes = [vp, i32, i32, u64, u64, vp, i32, vp]
        L.vs_allreduce_finalize_p2p.argtypes = [vp, i32, i32, u64, u64, i32, i32, vp, vp, ctypes.c_uint32, vp, i32, P(vs_result)]
        L.vs_indices_from_values.argtypes = [vp, i32, i32, u64, u64, vp, i32, i32, P(vs_result)]
        L.vs_fused_partials.argtypes = [vp, i32, u64, u64, vp, i32, vp, i32, P(vs_scale), i32, vp, i32, u64, u64, i32,
                                        vp, i32]
        L.vs_run_fused.argtypes = [vp, i32, u64, u64, vp, i32, vp, i32, P(vs_scale), i32, vp, i32, i32, P(vs_result)]
        L.vs_run_fused_p2p.argtypes = [vp, i32, u64, u64, vp, i32, vp, i32, P(vs_scale), i32, vp, i32, u64, u64, i32, i32, i32, vp, vp,
                                       ctypes.c_uint32, P(vs_result)]
        L.vs_ctx_reload_env.argtypes = [vp]
        L.vs_ctx_set_halton_mode.argtypes = [vp, i32]
        L.vs_halton_terms_mode.argtypes = [i32, u64, i32, vp, vp, vp, u64, P(u64)]
        L.vs_last_tail_ns.argtypes = [vp, i32, vp]
        L.vs_halton_arith_check.argtypes = [i32, i32]
        L.vs_ctx_set_timing.argtypes = [vp, i32]
        L.vs_sample_flat_shard.argtypes = [vp, i32, u64, u64, vp, i32, vp, i32, P(vs_scale), u64, u64, vp, i32]
        L.vs_reference_permutation.argtypes = [u64, ctypes.c_uint32, vp, vp, P(i32)]
        L.vs_measure_fp64_peak.argtypes = [vp, P(ctypes.c_double)]
        L.vs_last_kernel_ms.argtypes = [vp, P(ctypes.c_float)]
        L.vs_objective_outputs.argtypes = [i32, i32, vp, i32, P(i32)]
        L.vs_last_network_stats.argtypes = [vp, vp]
        _lib = L
        return _lib


def check(status):
    if status != VS_OK:
        err = VarsensError("libvarsens_b200: status %d: %s" % (status, lib().vs_last_error().decode()))
        err.status = status
        raise err


def objective_outputs(k, objective, params):
    """Outputs per point l of a registered objective (vs_objective_outputs: host only, validates the parameters).  Every
    objective but a mass-action network has one, known without a call."""
    if int(objective) not in (OBJ_MASS_ACTION, OBJ_MASS_ACTION_ADAPTIVE, OBJ_MASS_ACTION_STIFF):
        return 1
    par = numpy.ascontiguousarray(params, dtype=numpy.float64)
    l = ctypes.c_int()
    check(lib().vs_objective_outputs(int(k), int(objective), par.ctypes.data_as(ctypes.c_void_p), int(par.size), ctypes.byref(l)))
    return int(l.value)


def discard_arg(discard):
    """``discard`` as the C ABI takes it.  The ABI is unsigned: ctypes would wrap a negative value around 2^64 instead of
    refusing it, so it is rejected here."""
    d = int(discard)
    if d < 0:
        raise VarsensError("discard must be >= 0, got %d" % d)
    return d


def _is_torch_tensor(x):
    return type(x).__module__.startswith("torch") and hasattr(x, "data_ptr")


def buf(x, dtype=None, out=False):
    """(pointer, mem flag, keepalive) for a numpy array or torch tensor (None -> NULL).  ``out=True``: the library writes
    into the buffer, so a numpy array must already be C-contiguous and of the right dtype (a silent copy would be
    written instead of the caller's array)."""
    if x is None:
        return None, MEM_HOST, None
    if _is_torch_tensor(x):
        if not x.is_contiguous():
            raise VarsensError("tensor must be contiguous")
        if dtype is not None:
            import torch
            want = {numpy.float64: torch.float64, numpy.uint32: torch.int32}[dtype]
            if x.dtype not in (want, getattr(torch, "uint32", want)):
                raise VarsensError("tensor dtype %s, expected %s" % (x.dtype, want))
        return ctypes.c_void_p(x.data_ptr()), (MEM_DEVICE if x.is_cuda else MEM_HOST), x
    if out:
        if not isinstance(x, numpy.ndarray) or not x.flags.c_contiguous or not x.flags.writeable or \
                (dtype is not None and x.dtype != numpy.dtype(dtype)):
            raise VarsensError("output buffer must be a writeable C-contiguous numpy array of dtype %s (or a torch tensor)"
                               % (numpy.dtype(dtype).name if dtype is not None else "matching"))
        return x.ctypes.data_as(ctypes.c_void_p), MEM_HOST, x
    a = numpy.ascontiguousarray(x, dtype=dtype)
    return a.ctypes.data_as(ctypes.c_void_p), MEM_HOST, a


def _source_args(k, perm, raw, scale, params=None):
    """The design's source and objective parameters as the C ABI takes them: ((perm, perm_mem, raw, raw_mem, scale),
    (params, n_params) or () without params, the objects that must stay alive while the library reads them)."""
    sp, sk = scale.c_struct(k)
    pp, pm, pk = buf(perm, numpy.uint32)
    rp, rm, rk = buf(raw, numpy.float64)
    par = None if params is None else numpy.ascontiguousarray(params, dtype=numpy.float64)
    pa = () if par is None else (par.ctypes.data_as(ctypes.c_void_p), int(par.size))
    return (pp, pm, rp, rm, sp), pa, (sk, pk, rk, par)


def _peer_arrays(world, peer_bufs, peer_flags):
    """The uint64[world] tables of an exchange: every rank's buffer and every rank's flag array."""
    return tuple((ctypes.c_uint64 * world)(*[int(x) for x in a]) for a in (peer_bufs, peer_flags))


class Scale(object):
    """Host descriptor lowered to vs_scale (identity / linear / power)."""

    def __init__(self, kind=SCALE_IDENTITY, lower=None, upper=None):
        self.kind, self.lower, self.upper = kind, lower, upper

    def c_struct(self, k):
        if self.kind == SCALE_IDENTITY:
            return None, None
        lo = numpy.ascontiguousarray(numpy.broadcast_to(numpy.asarray(self.lower, dtype=numpy.float64), (k,)))
        up = numpy.ascontiguousarray(numpy.broadcast_to(numpy.asarray(self.upper, dtype=numpy.float64), (k,)))
        s = vs_scale(self.kind, lo.ctypes.data_as(ctypes.c_void_p), up.ctypes.data_as(ctypes.c_void_p))
        return ctypes.byref(s), (s, lo, up)

    def apply_numpy(self, p):
        """Same arithmetic on the host (used only to validate a traced scaling callable)."""
        if self.kind == SCALE_LINEAR:
            return p * (numpy.asarray(self.upper) - numpy.asarray(self.lower)) + numpy.asarray(self.lower)
        if self.kind == SCALE_POWER:
            return numpy.asarray(self.lower) * ((numpy.asarray(self.upper) / numpy.asarray(self.lower)) ** p)
        return p


IDENTITY = Scale()


class Result(object):
    """Host arrays shaped like the reference's attributes (varsens/saltelli.py:577-622)."""

    def __init__(self, k, l, second_order=True):
        self._view(k, l, numpy.zeros(_block_len(k, l, second_order)), second_order)

    def _view(self, k, l, flat, second_order):
        self.k, self.l = k, l
        self.sens_2 = self.sens_2n = None
        at = 0
        for name, cnt, shape in _result_fields(k, l, second_order):
            setattr(self, name, flat[at:at + cnt].reshape(shape))
            at += cnt
        return self

    @classmethod
    def views(cls, k, l, flat, second_order=True):
        """Result whose arrays are views of one flat float64 buffer in the library's result order (no copies)."""
        return cls.__new__(cls)._view(k, l, flat, second_order)

    @staticmethod
    def flat_len(k, l):
        return _block_len(k, l)

    @classmethod
    def from_flat(cls, k, l, flat, second_order=True):
        """Unpack the device result layout of vs_finalize_device (a host numpy copy of it)."""
        return cls.views(k, l, numpy.array(flat[:_block_len(k, l, second_order)], dtype=numpy.float64), second_order)

    def c_struct(self):
        """vs_result pointing at these arrays (NULL for the second-order arrays of a first-order result)."""
        arrays = [getattr(self, name) for name, _ in vs_result._fields_]
        return vs_result(*[None if a is None else a.ctypes.data for a in arrays])


class Context(object):
    """One vs_ctx per (process, device)."""

    _cache = {}

    def __init__(self, device=0):
        self._h = ctypes.c_void_p()
        check(lib().vs_ctx_create(int(device), ctypes.byref(self._h)))
        self.device = int(device)

    @classmethod
    def get(cls, device=None):
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
        if device not in cls._cache:
            cls._cache[device] = Context(device)
        return cls._cache[device]

    def close(self):
        if self._h:
            lib().vs_ctx_destroy(self._h)
            self._h = ctypes.c_void_p()

    @property
    def handle(self):
        return self._h

    def synchronize(self):
        check(lib().vs_ctx_synchronize(self._h))

    def set_stream(self, cuda_stream_ptr):
        """Run on a caller stream.  ``None`` = the ctx's own stream; ``0`` (torch's default stream handle) is mapped
        to cudaStreamLegacy (0x1) so that torch events on the default stream really bracket the kernels."""
        if cuda_stream_ptr is None:
            ptr = 0
        else:
            ptr = int(cuda_stream_ptr) or 1
        check(lib().vs_ctx_set_stream(self._h, ctypes.c_void_p(ptr)))
        self._stream_ptr = cuda_stream_ptr

    def reload_env(self):
        """Re-read the VS_* switches from the environment (they are otherwise read once, when the ctx is created)."""
        check(lib().vs_ctx_reload_env(self._h))

    def set_halton_mode(self, mode):
        """Arithmetic of the Halton radical inverse (HALTON_DIVIDE / _RECIPROCAL / _RUNNING_RECIPROCAL / _HORNER)."""
        check(lib().vs_ctx_set_halton_mode(self._h, int(mode)))

    def last_tail_ns(self, k):
        """ns spent in {combine+pack, peer stores, wait for peers, sum+estimators} by the tail of the last fused step."""
        a = numpy.zeros(11)
        check(lib().vs_last_tail_ns(self._h, int(k), a.ctypes.data_as(ctypes.c_void_p)))
        return a

    def launch_count(self):
        return int(lib().vs_ctx_launch_count(self._h))

    def network_stats(self):
        """Step counts of the last call that evaluated an adaptive mass-action network (vs_last_network_stats), over the rows
        it evaluated: {"accepted", "rejected", "failed" (trajectories), "lane_work"}.  (accepted + rejected) / lane_work is
        the share of warp lanes that did useful work."""
        a = numpy.zeros(4, dtype=numpy.uint64)
        check(lib().vs_last_network_stats(self._h, a.ctypes.data_as(ctypes.c_void_p)))
        return dict(zip(NETWORK_STATS, (int(v) for v in a)))

    def set_timing(self, on=True):
        """Record CUDA events around the main kernel of each call (read them with last_kernel_ms); off by default."""
        check(lib().vs_ctx_set_timing(self._h, int(bool(on))))

    def last_kernel_ms(self):
        ms = ctypes.c_float()
        check(lib().vs_last_kernel_ms(self._h, ctypes.byref(ms)))
        return float(ms.value)

    def measure_fp64_peak(self):
        t = ctypes.c_double()
        check(lib().vs_measure_fp64_peak(self._h, ctypes.byref(t)))
        return float(t.value)

    # ---- generators -----------------------------------------------------------------------
    def halton(self, k, first_index, count, scale=IDENTITY, out=None):
        out = numpy.empty((int(count), int(k))) if out is None else out
        sp, keep = scale.c_struct(k)
        op, om, _ = buf(out, numpy.float64, out=True)
        check(lib().vs_halton(self._h, int(k), int(first_index), int(count), sp, op, om))
        return out

    def sobol(self, k, first_point, count, dirnums, quantize6=False, scale=IDENTITY, out=None):
        out = numpy.empty((int(count), int(k))) if out is None else out
        d = numpy.ascontiguousarray(dirnums, dtype=numpy.uint32)
        if d.shape != (k, 32):
            raise VarsensError("dirnums must have shape (k, 32)")
        sp, keep = scale.c_struct(k)
        op, om, _ = buf(out, numpy.float64, out=True)
        check(lib().vs_sobol(self._h, int(k), int(first_point), int(count), d.ctypes.data_as(ctypes.c_void_p),
                             int(bool(quantize6)), sp, op, om))
        return out

    def sample_flat(self, k, n, perm, discard=0, scale=IDENTITY, raw=None, row_begin=0, row_end=None, out=None):
        total = 2 * n * (1 + k)
        row_end = total if row_end is None else row_end
        out = numpy.empty((int(row_end - row_begin), int(k))) if out is None else out
        src, _, keep = _source_args(k, perm, raw, scale)
        op, om, _ = buf(out, numpy.float64, out=True)
        check(lib().vs_sample_flat(self._h, int(k), int(n), discard_arg(discard), *src, int(row_begin), int(row_end), op, om))
        return out

    def sample_flat_shard(self, k, n, perm, i_begin, i_end, discard=0, scale=IDENTITY, raw=None, out=None):
        """Base rows [i_begin,i_end) of EVERY block of Sample.flat(): (2+2k, i_end-i_begin, k) -- a rank's share in multi-GPU
        export mode (vs_sample_flat_shard)."""
        rows = int(i_end - i_begin)
        out = numpy.empty((2 + 2 * int(k), rows, int(k))) if out is None else out
        src, _, keep = _source_args(k, perm, raw, scale)
        op, om, _ = buf(out, numpy.float64, out=True)
        check(lib().vs_sample_flat_shard(self._h, int(k), int(n), discard_arg(discard), *src, int(i_begin), int(i_end), op, om))
        return out

    # ---- objective values / estimators --------------------------------------------------------
    def eval_values(self, k, n, perm, objective, params, discard=0, scale=IDENTITY, raw=None, i_begin=0, i_end=None,
                    out=None):
        """(2+2k, rows) values, or (2+2k, rows, l) for an objective with l > 1 outputs (fvals[(t*rows + r)*l + o])."""
        i_end = n if i_end is None else i_end
        l = objective_outputs(k, objective, params)
        if out is None:
            out = numpy.empty((2 + 2 * k, int(i_end - i_begin)) + ((l,) if l > 1 else ()))
        src, par, keep = _source_args(k, perm, raw, scale, params)
        op, om, _ = buf(out, numpy.float64, out=True)
        check(lib().vs_eval_values(self._h, int(k), int(n), discard_arg(discard), *src, int(objective), *par, int(i_begin),
                                   int(i_end), op, om))
        return out

    def partials_from_values(self, k, l, rows, fvals, shift=None, flags=FLAG_SECOND_ORDER, out=None):
        plen = int(lib().vs_partials_len(int(k), int(l)))
        out = numpy.empty(plen) if out is None else out
        fp, fm, fk = buf(fvals, numpy.float64)
        sh = None if shift is None else numpy.ascontiguousarray(shift, dtype=numpy.float64)
        shp = None if sh is None else sh.ctypes.data_as(ctypes.c_void_p)
        op, om, _ = buf(out, numpy.float64, out=True)
        check(lib().vs_partials_from_values(self._h, int(k), int(l), int(rows), fp, fm, shp, int(flags), op, om))
        return out

    def finalize(self, k, l, n, partials, flags=FLAG_SECOND_ORDER, rows=None):
        res = Result(k, l, bool(flags & FLAG_SECOND_ORDER))
        cs = res.c_struct()
        pp, pm, pk = buf(partials, numpy.float64)
        check(lib().vs_finalize(self._h, int(k), int(l), int(n), int(n if rows is None else rows), pp, pm, int(flags),
                                ctypes.byref(cs)))
        return res

    def finalize_device(self, k, l, n, partials, out, flags=FLAG_SECOND_ORDER, rows=None):
        """vs_finalize_device: results stay in the CUDA tensor `out` (Result.from_flat unpacks a host copy); nothing syncs."""
        pp, pm, pk = buf(partials, numpy.float64)
        op, om, ok_ = buf(out, numpy.float64, out=True)
        if pm != MEM_DEVICE or om != MEM_DEVICE:
            raise VarsensError("finalize_device needs device tensors")
        check(lib().vs_finalize_device(self._h, int(k), int(l), int(n), int(n if rows is None else rows), pp, int(flags), op))
        return out

    def allreduce_finalize_p2p(self, k, l, n, world_size, rank, peer_bufs, peer_flags, epoch, partials, flags=FLAG_SECOND_ORDER,
                               rows=None):
        """All-reduce over NVLink peer memory fused with the finalisation (vs_allreduce_finalize_p2p)."""
        res = Result(k, l, bool(flags & FLAG_SECOND_ORDER))
        cs = res.c_struct()
        pb, pf = _peer_arrays(world_size, peer_bufs, peer_flags)
        pp, pm, pk = buf(partials, numpy.float64)
        if pm != MEM_DEVICE:
            raise VarsensError("partials must be a device tensor")
        check(lib().vs_allreduce_finalize_p2p(self._h, int(k), int(l), int(n), int(n if rows is None else rows), int(world_size),
                                              int(rank), pb, pf, int(epoch), pp, int(flags), ctypes.byref(cs)))
        return res

    def indices_from_values(self, k, l, n, rows, fvals, flags=FLAG_SECOND_ORDER):
        res = Result(k, l, bool(flags & FLAG_SECOND_ORDER))
        cs = res.c_struct()
        fp, fm, fk = buf(fvals, numpy.float64)
        check(lib().vs_indices_from_values(self._h, int(k), int(l), int(n), int(rows), fp, fm, int(flags),
                                           ctypes.byref(cs)))
        return res

    # ---- fused ------------------------------------------------------------------------------------
    def fused_partials(self, k, n, perm, objective, params, discard=0, scale=IDENTITY, raw=None, i_begin=0, i_end=None,
                       flags=FLAG_SECOND_ORDER, out=None):
        i_end = n if i_end is None else i_end
        plen = int(lib().vs_partials_len(int(k), objective_outputs(k, objective, params)))
        out = numpy.empty(plen) if out is None else out
        src, par, keep = _source_args(k, perm, raw, scale, params)
        op, om, _ = buf(out, numpy.float64, out=True)
        check(lib().vs_fused_partials(self._h, int(k), int(n), discard_arg(discard), *src, int(objective), *par, int(i_begin),
                                      int(i_end), int(flags), op, om))
        return out

    def run_fused(self, k, n, perm, objective, params, discard=0, scale=IDENTITY, raw=None, flags=FLAG_SECOND_ORDER):
        res = Result(k, objective_outputs(k, objective, params), bool(flags & FLAG_SECOND_ORDER))
        cs = res.c_struct()
        src, par, keep = _source_args(k, perm, raw, scale, params)
        check(lib().vs_run_fused(self._h, int(k), int(n), discard_arg(discard), *src, int(objective), *par, int(flags),
                                 ctypes.byref(cs)))
        return res

    def run_fused_p2p(self, k, n, perm, objective, params, world_size, rank, peer_bufs, peer_flags, epoch, i_begin, i_end,
                      discard=0, scale=IDENTITY, raw=None, flags=FLAG_SECOND_ORDER):
        """vs_run_fused_p2p: this rank's shard [i_begin,i_end) of the fused step, all-reduce over NVLink peer memory and
        estimators inside the ONE kernel launch; returns the Result (identical bits on every rank)."""
        res = Result(k, objective_outputs(k, objective, params), bool(flags & FLAG_SECOND_ORDER))
        cs = res.c_struct()
        src, par, keep = _source_args(k, perm, raw, scale, params)
        pb, pf = _peer_arrays(world_size, peer_bufs, peer_flags)
        check(lib().vs_run_fused_p2p(self._h, int(k), int(n), discard_arg(discard), *src, int(objective), *par, int(i_begin),
                                     int(i_end), int(flags), int(world_size), int(rank), pb, pf, int(epoch), ctypes.byref(cs)))
        return res

    def fused_plan(self, *args, **kwargs):
        """FusedPlan(self, *args, **kwargs): a fused step prepared once and run many times."""
        return FusedPlan(self, *args, **kwargs)


class FusedPlan(object):
    """A prepared fused step: every argument of vs_run_fused / vs_run_fused_p2p converted once (ctypes pointers, descriptor
    structs, peer tables), so that ``run()`` costs one foreign call -- the per-step host overhead matters once the GPU work is
    ~0.6 ms (8-GPU strong scaling of BASELINE config 3).  ``exchange`` = a dist.PeerExchange for the multi-GPU one-launch step
    (rows [i_begin, i_end) are this rank's shard), None for a single GPU.  The buffers passed in must stay alive and unchanged
    while the plan is used.  ``run()`` returns a Result whose arrays are views of one of the plan's TWO output buffers (used
    alternately): they stay valid until the run after the next one -- copy them to keep them longer.  (Allocating the buffer,
    the descriptor struct and the eight views per call cost 11 us of Python per step, 1.7 % of an 8-GPU step.)"""

    def __init__(self, ctx, k, n, perm, objective, params, discard=0, scale=IDENTITY, raw=None, flags=FLAG_SECOND_ORDER,
                 i_begin=0, i_end=None, exchange=None):
        self.ctx, self.k, self.second = ctx, int(k), bool(flags & FLAG_SECOND_ORDER)
        self.exchange = exchange
        src, par, self._keep = _source_args(k, perm, raw, scale, params)
        self.l = l = objective_outputs(k, objective, params)
        self._out = []                                   # two output sets: (byref of the vs_result struct, Result, struct)
        for _ in range(2):
            res = Result(self.k, l, self.second)
            cs = res.c_struct()
            self._out.append((ctypes.byref(cs), res, cs))
        self._turn = 0
        L = lib()
        i_end = n if i_end is None else i_end
        if exchange is None:
            if i_begin != 0 or i_end != n:
                raise VarsensError("a single-GPU plan covers the whole design")
            self._fn = L.vs_run_fused
            self._args = (ctx._h, int(k), int(n), discard_arg(discard), *src, int(objective), *par, int(flags))
        else:
            self._fn = L.vs_run_fused_p2p
            self._args = (ctx._h, int(k), int(n), discard_arg(discard), *src, int(objective), *par, int(i_begin), int(i_end),
                          int(flags), int(exchange.world), int(exchange.rank),
                          *_peer_arrays(exchange.world, exchange.peer_bufs, exchange.peer_flags))

    def run(self):
        self._turn ^= 1
        ref, res, _ = self._out[self._turn]
        if self.exchange is None:
            st = self._fn(*self._args, ref)
        else:
            st = self._fn(*self._args, self.exchange.next_epoch(), ref)
        if st != VS_OK:
            check(st)
        return res


def reference_permutation(n, seed=1):
    """(perm uint32[n], numpy legacy RNG state after the shuffle) of ``numpy.random.seed(seed); numpy.random.shuffle(rows)``
    (varsens/saltelli.py:100-101), computed by the library's own MT19937 (host code, no GPU needed)."""
    n = int(n)
    perm = numpy.empty(n, dtype=numpy.uint32)
    key = numpy.empty(624, dtype=numpy.uint32)
    pos = ctypes.c_int()
    check(lib().vs_reference_permutation(n, int(seed), perm.ctypes.data_as(ctypes.c_void_p), key.ctypes.data_as(ctypes.c_void_p),
                                         ctypes.byref(pos)))
    return perm, ("MT19937", key, int(pos.value), 0, 0.0)


def halton_terms(k, max_index, mode=HALTON_DIVIDE):
    """Host-only: the library's term table (bases, ndigits, offsets, terms) in one of the term-table modes."""
    L = lib()
    bases = numpy.zeros(k, dtype=numpy.uint32)
    check(L.vs_halton_bases(int(k), bases.ctypes.data_as(ctypes.c_void_p)))
    cnt = ctypes.c_uint64()
    nd = numpy.zeros(k, dtype=numpy.uint32)
    off = numpy.zeros(k, dtype=numpy.uint32)
    check(L.vs_halton_terms_mode(int(k), int(max_index), int(mode), nd.ctypes.data_as(ctypes.c_void_p),
                                 off.ctypes.data_as(ctypes.c_void_p), None, 0, ctypes.byref(cnt)))
    terms = numpy.zeros(int(cnt.value))
    check(L.vs_halton_terms_mode(int(k), int(max_index), int(mode), nd.ctypes.data_as(ctypes.c_void_p),
                                 off.ctypes.data_as(ctypes.c_void_p), terms.ctypes.data_as(ctypes.c_void_p),
                                 int(cnt.value), ctypes.byref(cnt)))
    return bases, nd, off, terms
