"""The fused kernel in steady state, against the long-double CPU oracle (cport.run) at the contract tolerance.

The fused kernel is persistent.  Each CTA's E-warps loop over 32-row batches and hand every batch to an S-warp through a
one-slot full/empty mbarrier pair, whose parity flips on each batch; after the loop the CTAs combine their partial sums in a
two-level ticket tail (groups of 16 CTAs, then the groups) and the last CTA computes the estimators (finalize_fixed<K>).
launch_fused_t sizes the grid so that each warp gets about one batch:
    variants 5 / 6:  CTAs = min(ceil(nbatch / E), SMs), E = 8 / 12 E-warps per CTA;
    variant 1:       CTAs = min(ceil(nbatch / 8), SMs), 8 warps per CTA;
so a run of a few thousand rows never reaches a warp's second batch, nor the second level of the tail.  The main size here is
N = 32 (38 SMs + 1) + 17 rows (180,017 on a 148-SM B200): nbatch = 38 SMs + 2, every variant runs one CTA per SM, each E-warp of
variant 6 takes 3 or 4 batches (4 in team 0 of CTA 0, 3 in its other teams), each warp of variants 5 and 1 takes 4 or 5, the
last batch has 17 rows, and the tail has ceil(SMs / 16) groups.

Every run at N asserts that it was in steady state, and fails (does not skip) otherwise: variants 5 and 6 run under VS_TRACE,
whose clock stamps of CTA 0 give each E-warp (warp id >= 4) its batch count -- there must be 8 or 12 E-warps, each with at least
three batches; variant 1 has no trace, its batches per warp follow from the formula above and the SM count.
  A. Every k from 2 to 20: the default route, variants 1 / 5 / 6 with and without the separable shortcut, first order, the
     Ishigami function; bit-identity where it holds by construction (a repeated call, and the tail's estimators against
     finalize_kernel on the same partial sums).
  B. The 32-bit index class, linear and power scaling, raw= points, the polled host permutation, ragged shards.
  C. Tail grid shapes from 1 CTA to one per SM, a last tail group of one CTA, and changing grids in one context.
  D. FusedPlan: the bits of run_fused, its two alternating output sets, interleaved plans.
  E. The one-rank peer exchange over successive epochs, directly and through a FusedPlan."""
import functools
import math

import numpy
import pytest

from conftest import close
from oracle import cport, pipeline

pytestmark = pytest.mark.gpu

A20 = [0, 0.5, 3, 9, 99, 99] + [99.0] * 14
NAMES = ("E_2", "var_y", "U_j", "U_nj", "sens", "sens_t", "sens_2", "sens_2n")
FIRST = NAMES[:6]
GF, ISHI = cport.OBJ_GFUNCTION, cport.OBJ_ISHIGAMI
SO, SEP = 1, 2                                       # FLAG_SECOND_ORDER, FLAG_SEPARABLE
TOP = 2 ** 32 - 1                                    # the largest Halton index a run may reach
WS_S, FUSED_WARPS = 4, 8                             # fused_impl.cuh: S-warps per CTA (variants 5, 6); warps of variant 1
EWARPS = {5: 8, 6: 12}                               # E-warps per CTA


@pytest.fixture(scope="module")
def vb():
    import varsens_b200
    return varsens_b200


@pytest.fixture(scope="module")
def ctx(vb):
    return vb.Context.get(0)


@pytest.fixture(scope="module")
def sms(ctx):
    import torch
    return torch.cuda.get_device_properties(ctx.device).multi_processor_count


def batches(rows):
    return -(-rows // 32)


@pytest.fixture(scope="module")
def N(sms):
    """nbatch = 38 SMs + 2: at least three batches for each of the 12 SMs E-warps of variant 6, the last batch ragged."""
    n = 32 * (38 * sms + 1) + 17
    assert batches(n) >= 3 * 12 * sms + 1 and n % 32 != 0
    return n


@functools.lru_cache(maxsize=None)
def perm_of(n):
    return pipeline.permutation(n).astype(numpy.uint32)


@functools.lru_cache(maxsize=64)
def oracle_gf(k, n):
    return cport.run(k, n, GF, gparams(k), perm=perm_of(n))


def gparams(k):
    return (A20 + [1.0, 2.0, 5.0, 99.0] * 30)[:k]


def disc(k, n, L):
    """discard whose run has the largest Halton index L."""
    return L - 20 * k - 2 * n


def grid_of(variant, rows, sms):
    """CTAs of the launch (launch_fused_t)."""
    per_cta = FUSED_WARPS if variant == 1 else EWARPS[variant]
    return max(1, min(-(-batches(rows) // per_cta), sms))


def form_of(k, flags, rows, variant=None, peer=False):
    """The variant that runs (fused_variant_for): 1 for first order; else VS_FUSED_VARIANT, or by default 6 below k = 20 and at
    k = 20 only for a generic single-GPU step of at least 2^22 rows."""
    if not flags & SO:
        return 1
    if variant is not None:
        return variant
    if k < 20:
        return 6
    return 6 if not flags & SEP and not peer and rows >= 1 << 22 else 5


def assert_indices(res, ref, names=NAMES, what=""):
    for name in names:
        try:
            close(numpy.asarray(getattr(res, name)).reshape(ref[name].shape), ref[name])
        except AssertionError as e:
            raise AssertionError("%s %s: %s" % (what, name, e))


def bits(a):
    return numpy.ascontiguousarray(a, dtype=numpy.float64).view(numpy.uint64)


def assert_bits(got, want, names=NAMES, what=""):
    for name in names:
        g, w = getattr(got, name), getattr(want, name)
        if w is None:
            assert g is None, (what, name)
        else:
            assert numpy.array_equal(bits(g), bits(w)), "%s %s: bits differ" % (what, name)


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


def e_warp_batches(path):
    """{E-warp id: batches} of CTA 0 from a VS_TRACE file: one line `warp it t0 t1 t2 t3` per batch `it` of an E-warp (warp
    id >= 4; the S-warps 0-3 number their lines differently)."""
    out = {}
    for line in path.read_text().splitlines():
        w, it = (int(x) for x in line.split()[:2])
        if w >= WS_S:
            out[w] = max(out.get(w, 0), it + 1)
    return out


def e_warp_schedule(variant, rows, sms):
    """{E-warp id: batches} of CTA 0 by fused_wsd_kernel's schedule: E-warp e of CTA b starts at batch
    (e / 4) 4 CTAs + 4 b + e % 4 and strides by E CTAs; warps without a batch leave no trace."""
    E, grid, nb = EWARPS[variant], grid_of(variant, rows, sms), batches(rows)
    first = {WS_S + e: (e // WS_S) * WS_S * grid + e % WS_S for e in range(E)}
    return {w: -(-(nb - b) // (E * grid)) for w, b in first.items() if b < nb}


class Runner(object):
    """Runs a fused call under VS_FUSED_VARIANT=variant (None: the default route) and checks the form that ran.  Variants 5 and
    6 are one launch and run under VS_TRACE: CTA 0's E-warps and their batch counts must be those of the form's schedule
    (8 or 12 E-warps when every one has a batch).  Variant 1 is several launches.  With steady (the default), every warp must
    also take at least three batches: E-warps by the trace, variant 1 by the host formula.  `counts` keeps the E-warp batch
    counts of the last traced call."""

    def __init__(self, ctx, monkeypatch, tmp_path, sms):
        self.ctx, self.mp, self.sms, self.trace = ctx, monkeypatch, sms, tmp_path / "trace.txt"
        self.counts = None

    def __call__(self, call, k, rows, flags=SO, variant=None, steady=True, peer=False, **env):
        form = form_of(k, flags, rows, variant, peer)
        what = "k %d rows %d flags %d variant %s (form %d)" % (k, rows, flags, variant, form)
        if self.trace.exists():
            self.trace.unlink()
        with switches(self.ctx, self.mp, VS_FUSED_VARIANT=variant, VS_TRACE=None if form == 1 else str(self.trace), **env):
            l0 = self.ctx.launch_count()
            res = call()
            launches = self.ctx.launch_count() - l0
        if form == 1:
            assert launches > 1, (what, launches)
            if steady:   # fused_kernel: warp w of CTA b takes batches 8 b + w, + 8 CTAs, ...
                least = batches(rows) // (FUSED_WARPS * grid_of(1, rows, self.sms))
                assert least >= 3, ("not in steady state", what, least)
        else:
            assert launches == 1, (what, launches)
            self.counts = e_warp_batches(self.trace)
            assert self.counts == e_warp_schedule(form, rows, self.sms), (what, self.counts)
            if steady:
                assert len(self.counts) == EWARPS[form], (what, sorted(self.counts))
                assert min(self.counts.values()) >= 3, ("not in steady state", what, self.counts)
        return res


@pytest.fixture
def run(ctx, monkeypatch, tmp_path, sms):
    return Runner(ctx, monkeypatch, tmp_path, sms)


# ------------------------------------------------------------------------------------------------
# A. every k, every form, against the oracle
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", (None, 1, 5, 6), ids=("default", "v1", "v5", "v6"))
@pytest.mark.parametrize("k", range(2, 21))
def test_fused_matrix(ctx, run, N, k, variant):
    """Second order with and without the separable shortcut under the default route (variant 6 below k = 20, 5 at k = 20: the
    rows are fewer than 2^22) or a forced variant; first order (always variant 1) with the v1 case.  Variants 5 and 6 also give
    the same bits twice -- the combine order is fixed, only which CTA runs the tail depends on timing -- and the tail's
    finalize_fixed<K> gives the bits of finalize_kernel (finalize_body) on the kernel's own partial sums."""
    a, p = gparams(k), perm_of(N)
    want = oracle_gf(k, N)
    for flags in (SO, SO | SEP):
        what = "variant %s flags %d" % (variant, flags)
        res = run(lambda: ctx.run_fused(k, N, p, GF, a, flags=flags), k, N, flags, variant)
        assert_indices(res, want, what=what)
        if form_of(k, flags, N, variant) == 6:
            assert sorted(set(run.counts.values())) == [3, 4], (what, run.counts)
        if variant in (5, 6):
            again = run(lambda: ctx.run_fused(k, N, p, GF, a, flags=flags), k, N, flags, variant)
            assert_bits(again, res, what=what + " repeated")
            part = run(lambda: ctx.fused_partials(k, N, p, GF, a, flags=flags), k, N, flags, variant)
            assert_bits(ctx.finalize(k, 1, N, part, flags=flags), res, what=what + " finalize_kernel vs the tail")
    if variant == 1:
        for flags in (0, SEP):
            res = run(lambda: ctx.run_fused(k, N, p, GF, a, flags=flags), k, N, flags)
            assert res.sens_2 is None and res.sens_2n is None
            assert_indices(res, want, FIRST, what="first order flags %d" % flags)


@pytest.mark.parametrize("variant", (1, 5, 6))
def test_fused_ishigami(ctx, run, N, variant):
    from varsens_b200 import _cabi
    k, par, pi = 3, [7.0, 0.1], math.pi
    sc = _cabi.Scale(_cabi.SCALE_LINEAR, numpy.full(k, -pi), numpy.full(k, pi))
    p = perm_of(N)
    want = cport.run(k, N, ISHI, par, scale=("linear", [-pi] * k, [pi] * k), perm=p)
    res = run(lambda: ctx.run_fused(k, N, p, ISHI, par, scale=sc), k, N, SO, variant)
    assert_indices(res, want, what="variant %d" % variant)


# ------------------------------------------------------------------------------------------------
# B. sources, index classes and shards
# ------------------------------------------------------------------------------------------------
def _each_wsd_form(ctx, run, k, n, want, **kw):
    """run_fused under variants 5 and 6, with and without the separable shortcut, against the oracle result `want`."""
    a, p = gparams(k), perm_of(n)
    for variant in (5, 6):
        for flags in (SO, SO | SEP):
            res = run(lambda: ctx.run_fused(k, n, p, GF, a, flags=flags, **kw), k, n, flags, variant)
            assert_indices(res, want, what="variant %d flags %d" % (variant, flags))


@pytest.mark.parametrize("k", (2, 9, 12, 16, 19))
def test_index_class_32(ctx, run, N, k):
    """Halton indices up to 2^32 - 1: the IB = 32 instantiations with the general-division digit positions."""
    discard = disc(k, N, TOP)
    _each_wsd_form(ctx, run, k, N, cport.run(k, N, GF, gparams(k), discard=discard, perm=perm_of(N)), discard=discard)


@pytest.mark.parametrize("k", range(2, 21))
def test_index_bits_32_bit_identical(ctx, run, N, k):
    """VS_INDEX_BITS=32 runs the IB = 32 instantiation of the same variant: the same additions in the same order, the extra
    digit positions add +0.0, so all eight outputs are bit-identical to the IB = 26 run."""
    a, p = gparams(k), perm_of(N)
    for variant in (5, 6):
        for flags in (SO, SO | SEP):
            base = run(lambda: ctx.run_fused(k, N, p, GF, a, flags=flags), k, N, flags, variant)
            wide = run(lambda: ctx.run_fused(k, N, p, GF, a, flags=flags), k, N, flags, variant, VS_INDEX_BITS=32)
            assert_bits(wide, base, what="variant %d flags %d" % (variant, flags))


@pytest.mark.parametrize("kind", ("linear", "power"))
@pytest.mark.parametrize("k", (5, 13, 17))
def test_scaling(ctx, run, N, k, kind):
    from varsens_b200 import _cabi
    lb, ub = numpy.linspace(0.1, 0.3, k), numpy.linspace(0.6, 0.95, k)
    sc = _cabi.Scale(_cabi.SCALE_LINEAR if kind == "linear" else _cabi.SCALE_POWER, lb, ub)
    discard = 2 ** 29 + 12345
    want = cport.run(k, N, GF, gparams(k), discard=discard, scale=(kind, lb, ub), perm=perm_of(N))
    _each_wsd_form(ctx, run, k, N, want, discard=discard, scale=sc)


@pytest.mark.parametrize("k", (4, 13, 20))
def test_raw_points(ctx, run, N, k):
    raw = numpy.random.RandomState(k).rand(2 * N, k)
    _each_wsd_form(ctx, run, k, N, cport.run(k, N, GF, gparams(k), raw=raw, perm=perm_of(N)), raw=raw)


@pytest.mark.parametrize("k", (2, 11, 13, 19))
def test_polled_host_permutation(ctx, run, k):
    """At >= 2^19 rows a host permutation is copied while the one launch runs, its lanes polling their entries: bit-identical
    to the device-permutation call, under the default variant and under variant 5."""
    import torch
    n = (1 << 19) + 17
    a, p = gparams(k), perm_of(n)
    pdev = torch.from_numpy(p.astype(numpy.int32)).cuda()
    for variant in (None, 5):
        dev = run(lambda: ctx.run_fused(k, n, pdev, GF, a), k, n, SO, variant)
        host = run(lambda: ctx.run_fused(k, n, p, GF, a), k, n, SO, variant)
        assert_bits(host, dev, what="variant %s" % variant)
        if variant is None:
            assert_indices(dev, oracle_gf(k, n))


@pytest.mark.parametrize("variant", (5, 6))
@pytest.mark.parametrize("k", (5, 14, 19))
def test_shards(ctx, run, N, k, variant):
    """Cuts inside a batch, a one-row shard and an empty one: the shards' partial sums add up to the whole run's."""
    a, p = gparams(k), perm_of(N)
    whole = run(lambda: ctx.fused_partials(k, N, p, GF, a), k, N, SO, variant)
    acc = numpy.zeros_like(whole)
    for lo, hi in ((0, 37889), (37889, 37890), (37890, 150001), (150001, N)):
        acc += run(lambda: ctx.fused_partials(k, N, p, GF, a, i_begin=lo, i_end=hi), k, hi - lo, SO, variant, steady=False)
    l0 = ctx.launch_count()
    empty = ctx.fused_partials(k, N, p, GF, a, i_begin=N, i_end=N)
    assert ctx.launch_count() == l0 and not empty.any()
    numpy.testing.assert_allclose(acc, whole, rtol=1e-13, atol=1e-12)
    assert_indices(ctx.finalize(k, 1, N, acc), oracle_gf(k, N))


# ------------------------------------------------------------------------------------------------
# C. tail grid shapes
# ------------------------------------------------------------------------------------------------
GRIDS = (1, 2, 15, 16, 17, 31, 32, 33, 147, 148)     # 16 CTAs per tail group: one group, a full one, a last group of one, ...


def tail_rows(variant, g):
    """Rows whose launch has exactly g CTAs: nbatch = E (g - 1) + 1 (ceil(nbatch / E) = g), the last batch of 7 rows."""
    return 32 * EWARPS[variant] * (g - 1) + 7


@pytest.mark.parametrize("g", GRIDS)
@pytest.mark.parametrize("k", (3, 12, 20))                # plain tile layout, paired layout, the shipped k
def test_tail_grid(ctx, run, sms, k, g):
    g = min(g, sms)
    a = gparams(k)
    for variant in (5, 6):
        n = tail_rows(variant, g)
        assert grid_of(variant, n, sms) == g
        p, want = perm_of(n), oracle_gf(k, n)
        for flags in (SO, SO | SEP):
            what = "variant %d grid %d flags %d" % (variant, g, flags)
            res = run(lambda: ctx.run_fused(k, n, p, GF, a, flags=flags), k, n, flags, variant, steady=False)
            assert_indices(res, want, what=what)
            part = run(lambda: ctx.fused_partials(k, n, p, GF, a, flags=flags), k, n, flags, variant, steady=False)
            assert_bits(ctx.finalize(k, 1, n, part, flags=flags), res, what=what + " finalize_kernel vs the tail")


@pytest.mark.parametrize("k", (12, 20))
def test_tail_grids_in_one_context(ctx, run, sms, k):
    """All SMs, 17 CTAs, 1 CTA, then again: every run resets the ticket counters it used and reuses block_buf, so each result
    has the bits of the first run of its grid."""
    a = gparams(k)
    for variant in (5, 6):
        first = {}
        for g in (148, 17, 1, 148, 17, 1):
            g = min(g, sms)
            n = tail_rows(variant, g)
            res = run(lambda: ctx.run_fused(k, n, perm_of(n), GF, a), k, n, SO, variant, steady=False)
            if g in first:
                assert_bits(res, first[g], what="variant %d grid %d" % (variant, g))
            else:
                first[g] = res


# ------------------------------------------------------------------------------------------------
# D. FusedPlan
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("flags", (SO, SO | SEP, 0), ids=("SO", "SO-SEP", "first"))
@pytest.mark.parametrize("k", (6, 20))
def test_fused_plan(ctx, run, N, k, flags):
    """plan.run() gives the bits of run_fused.  Its Result is a view of one of two output sets used alternately: the next run
    leaves it alone, the one after refills that same Result."""
    a, p = gparams(k), perm_of(N)
    names = NAMES if flags & SO else FIRST
    ref = ctx.run_fused(k, N, p, GF, a, flags=flags)
    plan = ctx.fused_plan(k, N, p, GF, a, flags=flags)
    r1 = run(plan.run, k, N, flags)
    assert_bits(r1, ref)
    kept = {name: getattr(r1, name).copy() for name in names}
    r2 = run(plan.run, k, N, flags)
    assert r2 is not r1
    assert_bits(r2, ref)
    for name in names:
        assert numpy.array_equal(bits(getattr(r1, name)), bits(kept[name])), name
        getattr(r1, name)[...] = numpy.nan
    r3 = run(plan.run, k, N, flags)
    assert r3 is r1
    assert_bits(r3, ref)


def test_fused_plans_interleaved(ctx, run, N):
    p = perm_of(N)
    args = {"A": (6, dict(flags=SO)), "B": (20, dict(flags=SO | SEP, discard=7))}
    plans = {key: ctx.fused_plan(k, N, p, GF, gparams(k), **kw) for key, (k, kw) in args.items()}
    refs = {key: ctx.run_fused(k, N, p, GF, gparams(k), **kw) for key, (k, kw) in args.items()}
    out = []
    for key in "ABA":
        k, kw = args[key]
        out.append((key, run(plans[key].run, k, N, kw["flags"])))
    for key, res in out:                                 # the first A is still valid: each plan has two output sets
        assert_bits(res, refs[key], what=key)


def test_single_gpu_plan_covers_the_design(ctx, vb, N):
    a, p = gparams(6), perm_of(N)
    for lo, hi in ((1, N), (0, N - 1)):
        with pytest.raises(vb.VarsensError, match="whole design"):
            ctx.fused_plan(6, N, p, GF, a, i_begin=lo, i_end=hi)


# ------------------------------------------------------------------------------------------------
# E. one-rank peer exchange over successive epochs
# ------------------------------------------------------------------------------------------------
DISCARDS = (0, 7, 0, 123)                            # epoch e writes set e % 2: epochs 3 and 4 reuse what 1 and 2 tagged


def exchange_buffer(k):
    """A zeroed exchange buffer of one rank: 2 sets x 1 slot x plen elements x 16 bytes (dist.PeerExchange)."""
    import torch
    m = 2 + 2 * k
    plen = 4 + m * (m + 1) // 2
    return torch.zeros(2 * 1 * plen * 2 + 16, dtype=torch.float64, device="cuda")


class OneRank(object):
    """The attributes of dist.PeerExchange that FusedPlan reads, for one rank (PeerExchange needs a process group)."""

    world, rank = 1, 0

    def __init__(self, buf):
        self.buf = buf
        self.peer_bufs = self.peer_flags = [buf.data_ptr()]
        self.epoch = 0

    def next_epoch(self):
        self.epoch += 1
        return self.epoch


@pytest.mark.parametrize("k", (6, 20))
def test_peer_exchange_epochs(ctx, run, N, k):
    """A one-rank vs_run_fused_p2p sums its own slot (0.0 + x = x) before the same estimators: the bits of run_fused at every
    epoch, though the inputs change from step to step."""
    a, p = gparams(k), perm_of(N)
    refs = {d: ctx.run_fused(k, N, p, GF, a, discard=d) for d in set(DISCARDS)}
    assert not numpy.array_equal(refs[0].sens, refs[7].sens)
    buf = exchange_buffer(k)
    ptr = [buf.data_ptr()]
    for epoch, d in enumerate(DISCARDS, 1):
        res = run(lambda: ctx.run_fused_p2p(k, N, p, GF, a, 1, 0, ptr, ptr, epoch, 0, N, discard=d), k, N, peer=True)
        assert_bits(res, refs[d], what="epoch %d discard %d" % (epoch, d))
    ex = OneRank(exchange_buffer(k))
    plans = {d: ctx.fused_plan(k, N, p, GF, a, discard=d, i_begin=0, i_end=N, exchange=ex) for d in set(DISCARDS)}
    for step, d in enumerate(DISCARDS, 1):
        res = run(plans[d].run, k, N, peer=True)
        assert ex.epoch == step
        assert_bits(res, refs[d], what="plan step %d discard %d" % (step, d))
