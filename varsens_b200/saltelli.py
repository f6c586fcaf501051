"""Host mirror of varsens/saltelli.py: Sample, Objective, Varsens with the reference's constructor
signatures, attribute names and shapes; every numerical step runs in libvarsens_b200.so on the GPU.

Differences from reference HEAD, all on the side of the *intended* API (SURVEY.md App. B):
  * ``Varsens(callable, scaling, k, n, verbose=...)`` works: ``verbose`` is passed by keyword
    (HEAD passes it into ``discard`` at saltelli.py:555 and into ``objective_vals`` at :567 -> TypeError).
  * ``M_1, M_2, N_j, N_nj`` (and ``fM_1 ...``) are materialised lazily, on first access: the fused
    path never builds them (the reference needs 2*k*n*k*8 bytes for N_j/N_nj, saltelli.py:119).
  * ``Sample(raw=...)`` does not shuffle the caller's array in place (HEAD quirk 5).
  * a one-observable value array may be 1-D (HEAD fails at :464 under numpy >= 2).
New optional keyword arguments (``device``) default to the reference behaviour.
"""
import os

import numpy

from . import _cabi, dist, functors, scale as _scale


def _say(verbose, *a, **kw):
    if verbose:
        print(*a, **kw)


_perm_cache = {}          # n -> (uint32 permutation, global numpy RNG state after drawing it); a few entries, newest last


def _reference_permutation(n):
    """The row order ``numpy.random.seed(1); numpy.random.shuffle(M_2)`` produces (saltelli.py:100-101), with the same side
    effect on numpy's global legacy RNG.  The Fisher-Yates walk is serial: numpy needs ~1 s for n = 2^24 (200x the GPU work
    that follows), the library's own MT19937 walk with look-ahead prefetching (vs_reference_permutation, bit-identical to
    numpy, tests/test_cabi_host.py) a fraction of that.  The order depends on n only (the seed is fixed), so the last few
    permutations are kept; a cache hit restores the RNG state the reference call would have left."""
    n = int(n)
    hit = _perm_cache.get(n)
    if hit is not None:
        numpy.random.set_state(hit[1])
        return hit[0]
    perm, state = _cabi.reference_permutation(n, 1)
    numpy.random.set_state(state)
    perm.setflags(write=False)
    while len(_perm_cache) >= 4:
        _perm_cache.pop(next(iter(_perm_cache)))
    _perm_cache[n] = (perm, state)
    return perm


_perm_dev_cache = {}      # (n, device) -> int32 CUDA tensor holding the same permutation; a few entries, newest last


def _device_permutation(perm, n, device):
    """The permutation as a device-resident tensor of GPU `device`, uploaded once per (n, device): the order depends on n only,
    so a repeated ``Varsens(functor, scaling, k, n)`` neither draws nor copies it again (64 MB over PCIe from pageable host
    memory cost as much as the whole fused step at n = 2^24).  Falls back to the host array when torch has no CUDA."""
    try:
        import torch
        if not torch.cuda.is_available():
            return perm
    except ImportError:
        return perm
    key = (int(n), int(device))
    t = _perm_dev_cache.get(key)
    if t is None:
        while len(_perm_dev_cache) >= 4:
            _perm_dev_cache.pop(next(iter(_perm_dev_cache)))
        t = torch.tensor(perm.view(numpy.int32), device=torch.device("cuda", int(device)))
        _perm_dev_cache[key] = t
    return t


class Sample(object):
    """Sample space definition plus the matrices M_1, M_2, N_j, N_nj (varsens/saltelli.py:13-250)."""

    def __init__(self, k, n, scaling=None, discard=0, verbose=True, raw=None, device=None, **loadArgs):
        self.k = int(k)
        self.n = int(n)
        self.scaling = scaling
        self.verbose = verbose
        self.discard = _cabi.discard_arg(discard)
        self._ctx = None
        self._device = device
        self._explicit = None        # (M_1, M_2, N_j, N_nj) given by a flattened file
        self._cache = {}
        self._raw = None
        self._perm = None
        self._scale = _cabi.IDENTITY

        if raw is not None:                                             # saltelli.py:69-73
            _say(verbose, "Using provided raw sample")
            x = numpy.asarray(raw)
            if x.shape != (2 * self.n, self.k):
                raise Exception("Raw sample dimensions do not match specified dimensions")
        elif loadArgs:                                                  # :74-77
            _say(verbose, "Loading Sample from loadArgs")
            x = self.load(**loadArgs)
            if x.shape == (2 * self.n * (1 + self.k), self.k):
                return
        else:                                                           # :78-84
            _say(verbose, "Generating Low Discrepancy Sequence")
            if not self.scaling:
                raise Exception("Generating a fresh sample space requires that a 'scaling' function be defined.")
            x = None

        if scaling is None:                                             # :86-88
            _say(verbose, "Defaulting to identity scaling of parameter space")
            self.scaling = lambda p: p

        desc = _scale.trace(self.scaling, self.k)
        if desc is not None:
            # scaling fused into the kernels; unscaled source is Halton (x is None) or the given block
            self._scale = desc
            self._raw = None if x is None else numpy.ascontiguousarray(x, dtype=numpy.float64)
        else:
            # arbitrary user callable: run it on the host on the two halves, as saltelli.py:92,95 do
            if x is None:
                x = self.ctx.halton(self.k, 20 * self.k + self.discard + 1, 2 * self.n)
            m1 = numpy.asarray(self.scaling(x[0:self.n, ...]), dtype=numpy.float64)
            m2 = numpy.asarray(self.scaling(x[self.n:2 * self.n, ...]), dtype=numpy.float64)
            self._raw = numpy.ascontiguousarray(numpy.concatenate((m1, m2), axis=0))
            self._scale = _cabi.IDENTITY
        _say(verbose, "Eliminating correlations")
        self._perm = _reference_permutation(self.n)                     # :100-101
        _say(verbose, "...Sample Created.")

    # ---- device plumbing ------------------------------------------------------------------
    @property
    def ctx(self):
        if self._ctx is None:
            self._ctx = _cabi.Context.get(self._device)
        return self._ctx

    def on_device(self):
        """True if rows can be generated by the kernels (not a flattened-file sample)."""
        return self._explicit is None

    def _perm_arg(self):
        """The row permutation as the kernels take it: the device-resident copy of this GPU (cached per n)."""
        if self._perm is None:
            return None
        return _device_permutation(self._perm, self.n, self.ctx.device)

    def flat_rows(self, row_begin, row_end, out=None):
        """Rows [row_begin,row_end) of flat(); `out` may be a CUDA torch tensor (stays on the GPU)."""
        if self._explicit is not None:
            return self._explicit_flat()[row_begin:row_end]
        return self.ctx.sample_flat(self.k, self.n, self._perm_arg(), self.discard, self._scale, self._raw,
                                    row_begin, row_end, out)

    def _block(self, name):
        if self._explicit is not None:
            return self._explicit[name]
        if name not in self._cache:
            n, k = self.n, self.k
            if name == "M_1":
                self._cache[name] = self.flat_rows(0, n)
            elif name == "M_2":
                self._cache[name] = self.flat_rows(n, 2 * n)
            elif name == "N_j":
                self._cache[name] = self.flat_rows(2 * n, 2 * n + k * n).reshape(k, n, k)
            else:
                self._cache[name] = self.flat_rows(2 * n + k * n, 2 * n + 2 * k * n).reshape(k, n, k)
        return self._cache[name]

    M_1 = property(lambda self: self._block("M_1"))
    M_2 = property(lambda self: self._block("M_2"))
    N_j = property(lambda self: self._block("N_j"))
    N_nj = property(lambda self: self._block("N_nj"))

    def generate_N_j(self, M_1, M_2):
        """k copies of M_2 with column i of copy i taken from M_1 (saltelli.py:112-125), built by the
        export-mode kernel from the two given (n,k) matrices."""
        M_1, M_2 = numpy.asarray(M_1, dtype=numpy.float64), numpy.asarray(M_2, dtype=numpy.float64)
        n, k = M_1.shape
        raw = numpy.ascontiguousarray(numpy.concatenate((M_1, M_2), axis=0))
        ident = numpy.arange(n, dtype=numpy.uint32)
        out = self.ctx.sample_flat(k, n, ident, 0, _cabi.IDENTITY, raw, 2 * n, 2 * n + k * n)
        return out.reshape(k, n, k)

    def _explicit_flat(self):
        if "flat" not in self._cache:                   # one concatenation, not one per window
            e = self._explicit
            self._cache["flat"] = numpy.concatenate([e["M_1"], e["M_2"]] + list(e["N_j"]) + list(e["N_nj"]), axis=0)
        return self._cache["flat"]

    def flat(self):
        """(2n(1+k), k): rows M_1 | M_2 | N_j[0..k) | N_nj[0..k) (saltelli.py:127-160)."""
        _say(self.verbose, "Flattening sample space...")
        x = self.flat_rows(0, 2 * self.n * (1 + self.k))
        _say(self.verbose, "...Done. ( flattened.shape = ", x.shape, ")")
        return x

    def export(self, outdir=os.getcwd(), prefix="sample", postfix=".txt", blocksize=float("inf"), delimiter="\t"):
        """Text batches ``prefix_{1..}postfix`` of `blocksize` flat rows (saltelli.py:173-193).  Blocks are
        generated window by window on the GPU, so the full flat matrix is never resident on the host.
        ``postfix=".npy"`` writes numpy binary batches instead of text (same names, same row windows)."""
        total = 2 * self.n * (1 + self.k)
        blocksize = total if blocksize > total else int(blocksize)
        prefix = _clean_prefix(outdir, prefix)
        nFiles = int(numpy.ceil(float(total) / blocksize))
        for b in range(nFiles):
            name = "%s%s" % (prefix, postfix) if nFiles == 1 else "%s_%d%s" % (prefix, b + 1, postfix)
            _say(self.verbose, "Writing to %s ..." % name, end=" ")
            _save_block(name, self.flat_rows(b * blocksize, min((b + 1) * blocksize, total)), delimiter)
            _say(self.verbose, "Done.")

    def load(self, indir='', loadFile=None, prefix=None, postfix='.txt', nFiles=None, offset=1, delimiter='\t'):
        """saltelli.py:195-250: a (2n,k) unscaled sample or a (2n(1+k),k) flattened scaled one."""
        files = _file_list("sample", "a sample", indir, loadFile, prefix, postfix, nFiles, offset)
        parts = []
        for f in files:
            _say(self.verbose, "Reading " + f + " ...", end=" ")
            parts.append(_load_block(f, delimiter, ndmin=2))
            _say(self.verbose, "Done.")
        x = numpy.vstack(parts)
        n, k = self.n, self.k
        if x.shape == (2 * n, k):
            if not self.scaling:
                raise Exception("Loading a pre-generated, unscaled sample space requires that a 'scaling' function be defined.")
        elif x.shape == (2 * n * (1 + k), k):
            _say(self.verbose, "Flattened sample detected")
            self._explicit = dict(M_1=x[0:n], M_2=x[n:2 * n],
                                  N_j=x[2 * n:2 * n + k * n].reshape(k, n, k).copy(),
                                  N_nj=x[2 * n + k * n:].reshape(k, n, k).copy())
        else:
            raise Exception("Loaded sample has shape " + str(x.shape) + ". Must have shape (%d,%d) or (%d,%d)."
                            % (2 * n, k, 2 * n * (1 + k), k))
        return x


def _is_binary(name):
    return str(name).endswith(".npy")


def _save_block(name, block, delimiter=" "):
    """One batch file: `%.18e` text exactly as the reference writes it (saltelli.py:190,411), or -- when the file name
    ends in .npy -- numpy's binary format (SURVEY.md §8f.2: bit-exact round trip, ~25x smaller and faster than text)."""
    if _is_binary(name):
        numpy.save(name, numpy.ascontiguousarray(block))
    else:
        numpy.savetxt(name, block, delimiter=delimiter)


def _load_block(name, delimiter=None, ndmin=0):
    if _is_binary(name):
        x = numpy.load(name)
        return numpy.atleast_2d(x) if ndmin == 2 and x.ndim < 2 else x
    with open(name, "rb") as fh:
        return numpy.loadtxt(fh, delimiter=delimiter, ndmin=ndmin)


def _clean_prefix(outdir, prefix):
    prefix = "_".join(str(prefix).split())
    if prefix[-1] == "_":
        prefix = prefix[:-1]
    return os.path.join(outdir, prefix)


def _file_list(noun, what, indir, loadFile, prefix, postfix, nFiles, offset):
    if loadFile:
        files = [os.path.join(indir, loadFile)]
    else:
        if not prefix:
            raise Exception("Either 'loadFile' or 'prefix' are required to load %s from file." % what)
        if not nFiles:
            raise Exception("Loading %s files with 'prefix' requires defining 'nFiles'." % noun)
        if prefix[-1] != "_":
            prefix += "_"
        files = [os.path.join(indir, prefix) + str(i) + postfix for i in range(offset, offset + nFiles)]
    for f in files:
        if not os.path.isfile(f):
            raise Exception("Cannot find input file " + f)
    return files


class Objective(object):
    """Objective values fM_1, fM_2 (n,l) and fN_j, fN_nj (k,n,l) (varsens/saltelli.py:252-495).

    ``objective_func`` may be
      * a registered device functor (varsens_b200.GFunction / Ishigami / RK4Chain / MassActionNetwork /
        AdaptiveMassActionNetwork): evaluated on the GPU; Varsens then uses the fused kernel (or the two-phase path) and
        these arrays are only built if you read them;
        a functor with l = outputs(k) > 1 outputs gives fM_1 (n, l), fN_j (k, n, l) and flat() (2n(1+k), l);
      * a callable marked with ``varsens_b200.vectorized``: gets CUDA tensors of sample rows;
      * any Python callable of one (k,) row, exactly as in the reference (called 2n(1+k) times).
    """

    def __init__(self, k, n, sample=None, objective_func=None, objective_vals=[], verbose=True, **loadArgs):
        self.k = k
        self.n = n
        self.sample = sample
        self.objective_func = objective_func
        self.verbose = verbose
        self._vals = None            # host (2n(1+k) [trimmed], l) flat values
        self._vals_dev = None        # same, CUDA torch tensor
        self._rows = n               # rows per block after NaN trimming
        self._functor = None
        _say(verbose, "Generating Objective Values.")
        if len(objective_vals) > 0:                                     # saltelli.py:297-298
            self.load(objective_vals)
        elif loadArgs:                                                  # :299-300
            self.load(**loadArgs)
        else:
            if not self.sample:                                         # :302-305
                raise Exception("Generating a fresh objective requires that a 'sample' be defined.")
            elif not self.objective_func:
                raise Exception("Generating a fresh objective requires that an 'objective_func' be defined.")
            if isinstance(objective_func, functors.Functor):
                if not sample.on_device():
                    raise Exception("Device functors need a generated or raw sample, not a flattened file")
                self._functor = objective_func          # evaluated lazily / fused by Varsens
            elif getattr(objective_func, "varsens_vectorized", False):
                self._evaluate_vectorized()
            else:
                self._evaluate_rows()

    # ---- evaluation routes ------------------------------------------------------------------
    def _evaluate_rows(self):
        """The reference's loop (saltelli.py:308-353): one Python call per sample row, in flat order."""
        f, n, k = self.objective_func, self.n, self.k
        total = 2 * n * (1 + k)
        step = max(1, 1 << 16)
        vals = None
        for r0 in range(0, total, step):
            rows = self.sample.flat_rows(r0, min(r0 + step, total))
            for i in range(rows.shape[0]):
                v = f(rows[i])
                if vals is None:
                    try:
                        l = len(v)
                    except TypeError:
                        l = 1
                    vals = numpy.zeros((total, l))
                vals[r0 + i] = v
        self._vals = vals

    def _evaluate_vectorized(self, max_bytes=1 << 28):
        import torch
        f, n, k = self.objective_func, self.n, self.k
        ctx = self.sample.ctx
        dev = torch.device("cuda", ctx.device)
        total = 2 * n * (1 + k)
        step = max(1, min(total, max_bytes // (8 * k)))
        block = torch.empty((step, k), dtype=torch.float64, device=dev)
        vals = None
        # The export-mode kernel and the user's torch code share `block`: run the ctx on torch's current stream for the
        # loop, so "generate window -> f(window) -> store -> generate next window" is ordered by the stream itself.
        with dist.on_torch_stream(ctx, dev):
            for r0 in range(0, total, step):
                r1 = min(r0 + step, total)
                view = block[:r1 - r0]
                if self.sample.on_device():
                    self.sample.flat_rows(r0, r1, out=view)
                else:                                   # flattened-file sample: the rows live on the host
                    view.copy_(torch.from_numpy(numpy.ascontiguousarray(self.sample.flat_rows(r0, r1), dtype=numpy.float64)))
                v = f(view)
                v = v.reshape(r1 - r0, -1).to(torch.float64)
                if vals is None:
                    vals = torch.empty((total, v.shape[1]), dtype=torch.float64, device=dev)
                vals[r0:r1] = v
        self._vals_dev = vals

    def _evaluate_functor(self):
        s = self.sample
        v = s.ctx.eval_values(self.k, self.n, s._perm_arg(), self._functor.objective_id, self._functor.params(self.k),
                              s.discard, s._scale, s._raw)
        self._functor.check_run(s.ctx)
        self._vals = numpy.ascontiguousarray(v.reshape(-1, self._functor.outputs(self.k)))

    def _host_vals(self):
        if self._vals is None:
            if self._vals_dev is not None:
                self._vals = self._vals_dev.cpu().numpy()
            elif self._functor is not None:
                self._evaluate_functor()
            else:
                return None
        return self._vals

    def _part(self, name):
        v = self._host_vals()
        if v is None:
            return None
        r, k = self._rows, self.k
        if name == "fM_1":
            return v[0:r]
        if name == "fM_2":
            return v[r:2 * r]
        if name == "fN_j":
            return v[2 * r:2 * r + k * r].reshape(k, r, -1)
        return v[2 * r + k * r:2 * r + 2 * k * r].reshape(k, r, -1)

    fM_1 = property(lambda self: self._part("fM_1"))
    fM_2 = property(lambda self: self._part("fM_2"))
    fN_j = property(lambda self: self._part("fN_j"))
    fN_nj = property(lambda self: self._part("fN_nj"))

    def flat(self):
        """(2n(1+k), l) in Sample.flat() row order (saltelli.py:357-391)."""
        return self._host_vals()

    def export(self, outdir=os.getcwd(), prefix="objective", postfix=".txt", blocksize=float("inf")):
        f = self.flat()                                                 # saltelli.py:393-413
        blocksize = len(f) if blocksize > len(f) else int(blocksize)
        prefix = _clean_prefix(outdir, prefix)
        nFiles = int(numpy.ceil(float(len(f)) / blocksize))
        for b in range(nFiles):
            name = "%s%s" % (prefix, postfix) if nFiles == 1 else "%s_%d%s" % (prefix, b + 1, postfix)
            _save_block(name, f[b * blocksize:(b + 1) * blocksize])

    def load(self, obj_vals=[], indir='', loadFile=None, prefix=None, postfix='.txt', nFiles=None, offset=1, scaling=1.0):
        """saltelli.py:415-495: values from an array or text files, `scaling` divisor (:451), NaN-row
        trimming over all four matrices (:474-495; the divisor n is NOT reduced, as in the reference)."""
        n, k = self.n, self.k
        if len(obj_vals) > 0:
            x = obj_vals
            if hasattr(x, "is_cuda"):
                x = x.detach().cpu().numpy()
        else:
            files = _file_list("objective", "an objective", indir, loadFile, prefix, postfix, nFiles, offset)
            obj = []
            for f in files:
                _say(self.verbose, "Reading " + f + " ...", end=" ")
                obj.append(_load_block(f))
                _say(self.verbose, "Done.")
            x = numpy.hstack(obj) if all(o.ndim <= 1 for o in obj) else numpy.vstack(obj)
        x = numpy.asarray(x, dtype=numpy.float64)
        if len(x) != 2 * n * (1 + k):
            raise Exception("Loaded objective has length " + str(len(x)) + ". Must have length %d." % (2 * n * (1 + k)))
        if x.ndim == 1:
            x = x.reshape(-1, 1)
        x = x / scaling
        # a base row is dropped from every block if any of its 2+2k values (first output) is NaN
        blocks = x.reshape(2 + 2 * k, n, -1)
        bad = numpy.isnan(blocks[:, :, 0]).any(axis=0)
        nbad = int(bad.sum())
        if nbad:
            blocks = blocks[:, ~bad, :]
            print("WARNING: %d of %d objectives were NaN, %f%% loss" % (nbad, 2 * n * (1 + k), 100.0 * nbad / (2 * n * (1 + k))))
        self._rows = n - nbad
        self._vals = numpy.ascontiguousarray(blocks.reshape((2 + 2 * k) * self._rows, -1))
        self._vals_dev = None


class Varsens(object):
    """Variance-based sensitivity by Saltelli's method (varsens/saltelli.py:497-628).

    Attributes after construction: ``E_2 (l,)``, ``var_y (l,)``, ``U_j, U_nj, sens, sens_t (k,l)``,
    ``sens_2, sens_2n (k,l,k,l)``."""

    def __init__(self, objective, scaling_func=None, k=None, n=None, sample=None, verbose=True):
        self.verbose = verbose
        if isinstance(sample, Sample):                                  # saltelli.py:548-551
            self.sample, self.k, self.n = sample, sample.k, sample.n
        elif k is not None and n is not None and scaling_func is not None:   # :552-555
            self.k, self.n = k, n
            self.sample = Sample(k, n, scaling_func, verbose=verbose)
        elif not isinstance(objective, Objective):                      # :556-559
            raise ValueError("Must specify sample, (k,n,scaling_func), or Objective object")
        if isinstance(objective, Objective):                            # :562-565
            self.objective, self.k, self.n = objective, objective.k, objective.n
        else:                                                           # :567 (intended keyword form)
            self.objective = Objective(self.k, self.n, self.sample, objective, verbose=verbose)
        self.compute_varsens()

    def compute_varsens(self):
        _say(self.verbose, "Final sensitivity calculation")
        o, k, n = self.objective, int(self.k), int(self.n)
        flags = _cabi.FLAG_SECOND_ORDER
        if o._functor is not None and o._vals is None and o._vals_dev is None:
            res = self._fused(o, k, n, flags)
        elif o._vals_dev is not None:
            ctx = o.sample.ctx if o.sample is not None else _cabi.Context.get()
            res = ctx.indices_from_values(k, o._vals_dev.shape[1], n, o._rows, o._vals_dev, flags)
        else:
            v = o._host_vals()
            ctx = o.sample.ctx if isinstance(o.sample, Sample) else _cabi.Context.get()
            res = ctx.indices_from_values(k, v.shape[1], n, o._rows, v, flags)
        for name in ("E_2", "var_y", "U_j", "U_nj", "sens", "sens_t", "sens_2", "sens_2n"):
            setattr(self, name, getattr(res, name))

    def _fused(self, o, k, n, flags):
        s, f = o.sample, o._functor
        res = dist.fused_step(s.ctx, k, n, s._perm_arg(), f.objective_id, f.params(k), s.discard, s._scale, s._raw, flags)
        f.check_run(s.ctx)
        return res
