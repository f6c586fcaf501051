"""Every form of the kernels the library selects between at run time, against the CPU oracle, at Halton indices up to 2^32 - 1.

The parity suite runs the default route of each entry point with indices below 2^25.  Here:
  A. the fused kernel across its index classes (IB = 26 / IB = 32 with and without the run-time `small` branch of
     halton_group) and across digit-count boundaries, in every variant (VS_FUSED_VARIANT = 1, 5, 6) and flag set;
  B. every fused variant for every k the fused route covers (2 ... 20), with proof that the forced variant really ran;
  C. the run-time-base generators of export mode and product-form evaluation at indices that need the general-division
     prologue (DimLoop::jg = 1, 2, 3);
  D. the other Halton arithmetics (vs_halton_mode 1 - 3) through the fused pipeline;
  E. range checks on `discard` (no Halton index may wrap around to 0).
References: cport.run at the contract tolerance (close), cport.sample_flat bit-exact, cport.values at rtol = 1e-13.
Runs are named by their LARGEST Halton index L = 20k + discard + 2n; a straddle of P puts the A indices at P - n ... P - 1 and
the B indices at P ... P + n - 1."""
import math

import numpy
import pytest

from conftest import close
from oracle import cport, halton as ohalton, pipeline

pytestmark = pytest.mark.gpu

A6 = [0, 0.5, 3, 9, 99, 99]
A20 = A6 + [99.0] * 14
NAMES = ("E_2", "var_y", "U_j", "U_nj", "sens", "sens_t", "sens_2", "sens_2n")
FIRST = NAMES[:6]
GF, ISHI, RK4 = cport.OBJ_GFUNCTION, cport.OBJ_ISHIGAMI, cport.OBJ_RK4_CHAIN
SO, SEP = 1, 2                                       # FLAG_SECOND_ORDER, FLAG_SEPARABLE
ERR_RANGE = 3
TOP = 2 ** 32 - 1                                    # the largest Halton index a run may reach


@pytest.fixture(scope="module")
def vb():
    import varsens_b200
    return varsens_b200


@pytest.fixture(scope="module")
def ctx(vb):
    return vb.Context.get(0)


def perm_of(n):
    return pipeline.permutation(n).astype(numpy.uint32)


def assert_indices(res, ref, names=NAMES, what=""):
    for name in names:
        try:
            close(numpy.asarray(getattr(res, name)).reshape(ref[name].shape), ref[name])
        except AssertionError as e:
            raise AssertionError("%s %s: %s" % (what, name, e))


def disc(k, n, L):
    """discard whose run has the largest Halton index L."""
    return L - 20 * k - 2 * n


def straddle(k, n, P):
    """discard whose A indices end at P - 1 and whose B indices start at P."""
    return P - n - 20 * k - 1


def gparams(k):
    return (A20 + [1.0, 2.0, 5.0, 99.0] * 30)[:k]


class switches(object):
    """VS_* switches for the body of a with-block (None = leave unset); afterwards every switch and the Halton mode are back
    at their defaults."""

    def __init__(self, ctx, monkeypatch, **env):
        self.ctx, self.mp, self.env = ctx, monkeypatch, {key: val for key, val in env.items() if val is not None}

    def __enter__(self):
        for key, val in self.env.items():
            self.mp.setenv(key, str(val))
        self.ctx.reload_env()
        return self

    def __exit__(self, *exc):
        for key in self.env:
            self.mp.delenv(key, raising=False)
        self.ctx.reload_env()
        self.ctx.set_halton_mode(0)
        return False


def _linear(k):
    from varsens_b200 import _cabi
    lb, ub = numpy.linspace(0.1, 0.3, k), numpy.linspace(0.6, 0.95, k)
    return _cabi.Scale(_cabi.SCALE_LINEAR, lb, ub), ("linear", lb, ub)


def fused_case(name):
    """(k, objective, params, scale, oracle scale) of a case of part A."""
    from varsens_b200 import _cabi
    if name == "ishigami":
        pi = math.pi
        return 3, ISHI, [7.0, 0.1], _cabi.Scale(_cabi.SCALE_LINEAR, numpy.full(3, -pi), numpy.full(3, pi)), ("linear", [-pi] * 3, [pi] * 3)
    if name == "g6lin":
        return (6, GF, gparams(6)) + _linear(6)
    k = int(name[1:])
    return k, GF, gparams(k), _cabi.IDENTITY, None


# class edges of the fused kernel: IB = 26 below 2^26, FusedConst::small_index below 2^29, the largest 32-bit index
EDGES = (2 ** 26 - 1, 2 ** 26, 2 ** 29 - 1, 2 ** 29, TOP)
# digit-count boundaries (P, smallest k with that base): base 2 gains its 32nd digit, base 3 its 21st, base 7 its 12th,
# base 23 its 8th, base 37 (the first computed-term base) its 7th -- the last constant row AR_J - 1
STRADDLES = ((2 ** 31, 1), (3 ** 20, 2), (7 ** 11, 1), (23 ** 7, 9), (37 ** 6, 12))


def _index_class_params():
    out = []
    for case in ("g3", "g6", "g12", "g20", "ishigami"):
        k = 3 if case == "ishigami" else int(case[1:])
        for n in (333, 2048):
            out += [pytest.param(case, n, "L", L, id="%s-n%d-L%d" % (case, n, L)) for L in EDGES]
            out += [pytest.param(case, n, "P", P, id="%s-n%d-P%d" % (case, n, P)) for P, kmin in STRADDLES if k >= kmin]
    out += [pytest.param("g6lin", n, "L", TOP, id="g6lin-n%d-L%d" % (n, TOP)) for n in (333, 2048)]
    return out


# ------------------------------------------------------------------------------------------------
# A. fused kernel across the index classes
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case,n,kind,at", _index_class_params())
def test_fused_index_classes(ctx, monkeypatch, case, n, kind, at):
    """Every fused variant (default, 1, 5, 6 -- each has its own IB = 32 instantiation) and flag set at the class edges of the
    digit code and across digit-count boundaries of the bases."""
    k, obj, par, sc, osc = fused_case(case)
    discard = disc(k, n, at) if kind == "L" else straddle(k, n, at)
    p = perm_of(n)
    want = cport.run(k, n, obj, par, discard=discard, scale=osc)
    for variant in (None, 1, 5, 6):
        with switches(ctx, monkeypatch, VS_FUSED_VARIANT=variant):
            for flags in ((SO, SO | SEP) if obj == GF else (SO,)):
                res = ctx.run_fused(k, n, p, obj, par, discard=discard, scale=sc, flags=flags)
                assert_indices(res, want, what="variant %s flags %d" % (variant, flags))


@pytest.mark.parametrize("k", range(2, 21))
def test_index_bits_32_is_bit_identical_below_2p26(ctx, monkeypatch, k):
    """VS_INDEX_BITS=32 runs the IB = 32 instantiation of the same variant: the same additions in the same order, the extra
    digit positions add +0.0, so all eight outputs are bit-identical to the IB = 26 run."""
    n = 333
    a, p = gparams(k), perm_of(n)
    discard = disc(k, n, 2 ** 26 - 1)
    base = ctx.run_fused(k, n, p, GF, a, discard=discard)
    with switches(ctx, monkeypatch, VS_INDEX_BITS=32):
        wide = ctx.run_fused(k, n, p, GF, a, discard=discard)
    for name in NAMES:
        assert (getattr(wide, name) == getattr(base, name)).all(), name


def test_fused_shards_at_the_largest_index(ctx):
    k, n = 20, 2048
    a, p = gparams(k), perm_of(n)
    discard = disc(k, n, TOP)
    whole = ctx.fused_partials(k, n, p, GF, a, discard=discard)
    acc = numpy.zeros_like(whole)
    for lo, hi in ((0, 700), (700, 701), (701, n)):
        acc += ctx.fused_partials(k, n, p, GF, a, discard=discard, i_begin=lo, i_end=hi)
    numpy.testing.assert_allclose(acc, whole, rtol=1e-13, atol=1e-12)
    assert_indices(ctx.finalize(k, 1, n, acc), cport.run(k, n, GF, a, discard=discard))


def test_fused_host_permutation_at_the_largest_index(ctx):
    """The polled host-permutation launch (>= 2^19 rows) in the IB = 32 class is bit-identical to the device-permutation one."""
    import torch
    k, n = 6, (1 << 19) + 5
    a, p = gparams(k), perm_of(n)
    discard = disc(k, n, TOP)
    l0 = ctx.launch_count()
    dev = ctx.run_fused(k, n, torch.from_numpy(p.astype(numpy.int32)).cuda(), GF, a, discard=discard)
    assert ctx.launch_count() - l0 == 1
    l0 = ctx.launch_count()
    host = ctx.run_fused(k, n, p, GF, a, discard=discard)
    assert ctx.launch_count() - l0 == 1
    for name in NAMES:
        assert (getattr(host, name) == getattr(dev, name)).all(), name
    assert_indices(dev, cport.run(k, n, GF, a, discard=discard, perm=p))


# ------------------------------------------------------------------------------------------------
# B. fused variant matrix
# ------------------------------------------------------------------------------------------------
def _trace_warps(path):
    with open(path) as f:
        return {int(line.split()[0]) for line in f if line.strip()}


def _run_forced(ctx, monkeypatch, tmp_path, variant, flags, run):
    """run() under VS_FUSED_VARIANT=variant; checks that the variant ran.  Variants 5 and 6 are one launch each; which of the
    two ran shows in the warp ids of CTA 0's clock stamps (VS_TRACE): 4 S-warps plus 8 (variant 5) or 12 (variant 6) E-warps,
    every one of which owns a batch when the run has at least 64 batches of 32 rows.  Variant 1 is several launches."""
    trace = str(tmp_path / "trace.txt") if variant in (5, 6) else None
    with switches(ctx, monkeypatch, VS_FUSED_VARIANT=variant, VS_TRACE=trace):
        l0 = ctx.launch_count()
        res = run()
        launches = ctx.launch_count() - l0
    if variant == 1:
        assert launches > 1, (variant, flags, launches)
    else:
        assert launches == 1, (variant, flags, launches)
        warps = _trace_warps(trace)
        assert len(warps) == 4 * (3 if variant == 5 else 4), (variant, flags, sorted(warps))
    return res


@pytest.mark.parametrize("n", (333, 2048))
@pytest.mark.parametrize("k", range(2, 21))
def test_fused_variant_matrix(ctx, monkeypatch, tmp_path, k, n):
    a, p = gparams(k), perm_of(n)
    want = cport.run(k, n, GF, a)
    for variant in (1, 5, 6):
        for flags in (SO, SO | SEP):
            if variant in (5, 6) and n < 2048:             # fewer batches than E-warps in CTA 0: no trace check
                with switches(ctx, monkeypatch, VS_FUSED_VARIANT=variant):
                    l0 = ctx.launch_count()
                    res = ctx.run_fused(k, n, p, GF, a, flags=flags)
                    assert ctx.launch_count() - l0 == 1
            else:
                res = _run_forced(ctx, monkeypatch, tmp_path, variant, flags, lambda: ctx.run_fused(k, n, p, GF, a, flags=flags))
            assert_indices(res, want, what="variant %d flags %d" % (variant, flags))
    first = ctx.run_fused(k, n, p, GF, a, flags=0)
    assert first.sens_2 is None and first.sens_2n is None
    assert_indices(first, want, FIRST, what="first order")


@pytest.mark.parametrize("n", (333, 2048))
def test_fused_ishigami_variants(ctx, monkeypatch, tmp_path, n):
    k, obj, par, sc, osc = fused_case("ishigami")
    p = perm_of(n)
    want = cport.run(k, n, obj, par, scale=osc)
    for variant in (1, 5, 6):
        if variant in (5, 6) and n < 2048:
            with switches(ctx, monkeypatch, VS_FUSED_VARIANT=variant):
                res = ctx.run_fused(k, n, p, obj, par, scale=sc)
        else:
            res = _run_forced(ctx, monkeypatch, tmp_path, variant, SO, lambda: ctx.run_fused(k, n, p, obj, par, scale=sc))
        assert_indices(res, want, what="variant %d" % variant)


# ------------------------------------------------------------------------------------------------
# C. export and evaluation generators at large indices
# ------------------------------------------------------------------------------------------------
LARGE = (pytest.param("L", 2 ** 29, id="L2^29"), pytest.param("L", TOP, id="L2^32-1"),
         pytest.param("P", 3 ** 20, id="P3^20"), pytest.param("P", 37 ** 6, id="P37^6"))
EXPORT_FORMS = ({}, {"VS_EXPORT_SLOW_GEN": 1}, {"VS_EXPORT_SLOW_GEN": 2}, {"VS_NO_BULK_EXPORT": 1})


@pytest.mark.parametrize("kind,at", LARGE)
@pytest.mark.parametrize("k", (7, 12, 50))
def test_sample_flat_large_indices(ctx, monkeypatch, k, kind, at):
    """Export mode (bulk-store kernel for even k, scalar-store kernel for odd k or VS_NO_BULK_EXPORT; multiply-only digit loop
    with computed terms, VS_EXPORT_SLOW_GEN=2, or the generic loop, =1) bit-exact where the leading digit positions need the
    general division: base 3 at 2^32 - 1 needs three such positions."""
    from varsens_b200 import _cabi
    n = 333
    discard = disc(k, n, at) if kind == "L" else straddle(k, n, at)
    p = perm_of(n)
    whole = cport.sample_flat(k, n, discard)
    total = 2 * n * (1 + k)
    blocks = whole.reshape(2 + 2 * k, n, k)
    for env in EXPORT_FORMS:
        with switches(ctx, monkeypatch, **env):
            assert (ctx.sample_flat(k, n, p, discard) == whole).all(), env
            for lo, hi in ((n - 3, n + 5), (2 * n + 7, 5 * n + 8), ((k + 1) * n - 1, (k + 3) * n + 2), (total - 33, total)):
                assert (ctx.sample_flat(k, n, p, discard, row_begin=lo, row_end=hi) == whole[lo:hi]).all(), (env, lo, hi)
            lo, hi = n // 3, n // 3 + 45
            assert (ctx.sample_flat_shard(k, n, p, lo, hi, discard) == blocks[:, lo:hi, :]).all(), env
    if k == 12 and at == TOP:
        sc, osc = _linear(k)
        assert (ctx.sample_flat(k, n, p, discard, sc) == cport.sample_flat(k, n, discard, scale=osc)).all()


@pytest.mark.parametrize("kind,at", (pytest.param("L", TOP, id="L2^32-1"), pytest.param("P", 37 ** 6, id="P37^6")))
@pytest.mark.parametrize("k", (24, 50, 100))
def test_eval_values_product_form_large_indices(ctx, k, kind, at):
    n = 333
    a, p = gparams(k), perm_of(n)
    discard = disc(k, n, at) if kind == "L" else straddle(k, n, at)
    got = ctx.eval_values(k, n, p, GF, a, discard=discard)
    numpy.testing.assert_allclose(got, cport.values(k, n, GF, a, discard=discard), rtol=1e-13, atol=0)
    if k == 24 and at == TOP:                                  # indices through the whole two-phase path
        assert_indices(ctx.run_fused(k, n, p, GF, a, discard=discard), cport.run(k, n, GF, a, discard=discard))


@pytest.mark.parametrize("kind,at", (pytest.param("L", TOP, id="L2^32-1"), pytest.param("P", 37 ** 6, id="P37^6")))
def test_eval_values_other_kernels_large_indices(ctx, monkeypatch, kind, at):
    """k = 6 by the product-form and the point-by-point kernel (VS_NO_PF_EVAL=1); the RK4 chain with linear scaling, whose
    trajectories are bit-identical to the oracle's when the rate constants are (test_eval_values_and_rk4)."""
    from varsens_b200 import _cabi
    k, n = 6, 333
    a, p = gparams(k), perm_of(n)
    discard = disc(k, n, at) if kind == "L" else straddle(k, n, at)
    want = cport.values(k, n, GF, a, discard=discard)
    for env in ({}, {"VS_NO_PF_EVAL": 1}):
        with switches(ctx, monkeypatch, **env):
            numpy.testing.assert_allclose(ctx.eval_values(k, n, p, GF, a, discard=discard), want, rtol=1e-13, atol=0, err_msg=str(env))
    k, n = 20, 64
    discard = disc(k, n, at) if kind == "L" else straddle(k, n, at)
    r = numpy.linspace(0.5, 2.0, k)
    got = ctx.eval_values(k, n, perm_of(n), RK4, [0.02, 250], discard=discard,
                          scale=_cabi.Scale(_cabi.SCALE_LINEAR, r * 0.5, r * 2))
    want = cport.values(k, n, RK4, [0.02, 250], discard=discard, scale=("linear", r * 0.5, r * 2))
    assert (got == want).all(), "%d of %d trajectories differ" % (int((got != want).sum()), got.size)


# ------------------------------------------------------------------------------------------------
# D. Halton modes through the fused pipeline
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("L", (None, TOP), ids=("small", "L2^32-1"))
@pytest.mark.parametrize("k", (6, 20))
@pytest.mark.parametrize("mode", (1, 2, 3))
def test_halton_modes_through_fused(ctx, monkeypatch, mode, k, L):
    """Modes 1 and 2 change the fused kernel's fixed table and computed-term constants; mode 3 (Horner) has no table and sends
    vs_run_fused to the two-phase path.  Reference: the oracle's restatement of that arithmetic as the unscaled points."""
    n = 1000
    a, p = gparams(k), perm_of(n)
    discard = 0 if L is None else disc(k, n, L)
    raw = ohalton.halton_points_mode(k, 20 * k + discard + 1, 2 * n, ohalton.MODES[mode])
    want = cport.run(k, n, GF, a, raw=raw)
    with switches(ctx, monkeypatch):
        ctx.set_halton_mode(mode)
        l0 = ctx.launch_count()
        res = ctx.run_fused(k, n, p, GF, a, discard=discard)
        launches = ctx.launch_count() - l0
        assert_indices(res, want)
        if mode == 3:
            assert launches > 1
            numpy.testing.assert_allclose(ctx.eval_values(k, n, p, GF, a, discard=discard), cport.values(k, n, GF, a, raw=raw),
                                          rtol=1e-13, atol=0)
        else:
            assert launches == 1


# ------------------------------------------------------------------------------------------------
# E. discard range
# ------------------------------------------------------------------------------------------------
def test_discard_range_is_checked_on_every_entry_point(ctx, vb):
    """A Halton index of 2^32 and a discard that would wrap the first index around 2^64 to 0 are refused (VS_ERR_RANGE) before
    anything is launched; a negative discard is refused by the binding (the C ABI is unsigned)."""
    k, n = 6, 64
    p = perm_of(n)
    calls = {
        "run_fused": lambda d: ctx.run_fused(k, n, p, GF, A6, discard=d),
        "fused_partials": lambda d: ctx.fused_partials(k, n, p, GF, A6, discard=d),
        "run_fused_p2p": lambda d: ctx.run_fused_p2p(k, n, p, GF, A6, 1, 0, [0], [0], 1, 0, n, discard=d),
        "eval_values": lambda d: ctx.eval_values(k, n, p, GF, A6, discard=d),
        "sample_flat": lambda d: ctx.sample_flat(k, n, p, d),
        "sample_flat_shard": lambda d: ctx.sample_flat_shard(k, n, p, 0, n, d),
    }
    l0 = ctx.launch_count()
    for name, call in calls.items():
        for d in (disc(k, n, 2 ** 32), 2 ** 64 - 20 * k - 1, 2 ** 32, 2 ** 64 - 1):
            with pytest.raises(vb.VarsensError) as e:
                call(d)
            assert e.value.status == ERR_RANGE, (name, d)
        with pytest.raises(vb.VarsensError, match="discard"):
            call(-1)
    assert ctx.launch_count() == l0
    assert_indices(ctx.run_fused(k, n, p, GF, A6, discard=disc(k, n, TOP)), cport.run(k, n, GF, A6, discard=disc(k, n, TOP)))
