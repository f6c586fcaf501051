"""GPU checks of the adaptive mass-action network objective (VS_OBJ_MASS_ACTION_ADAPTIVE, network_adaptive_kernel): values
and step counts bit for bit against the oracle's restatement (oracle/mass_action.c) in the 64- and 32-thread forms, past
the first CTA; rejections and failures; indices through the two-phase route; the Python API; the limits.

Every launch checked against its VS_TRACE line has at least 8 CTAs and a ragged last one (n = 8 nthr + 37)."""
import numpy
import pytest

from conftest import close
from oracle import exact as oexact, mass_action as ob
from test_gpu_mass_action import bits_equal, perm_of
from test_gpu_steady_state import Tracer
from test_gpu_value_kernels import differ, guarded, launch_line, net_smem, net_threads, optin
from varsens_b200._cabi import OBJ_MASS_ACTION_ADAPTIVE

pytestmark = pytest.mark.gpu

NAMES = ("E_2", "var_y", "U_j", "U_nj", "sens", "sens_t", "sens_2", "sens_2n")
MAA = OBJ_MASS_ACTION_ADAPTIVE
ERR_ARG, ERR_UNSUPPORTED = 1, 5
STATS = ("accepted", "rejected", "failed", "lane_work")


@pytest.fixture(scope="module")
def vb():
    import varsens_b200
    return varsens_b200


@pytest.fixture(scope="module")
def ctx(vb):
    return vb.Context.get(0)


def assert_form(lines, par, k, rows, nthr):
    f = launch_line(lines, "network_adaptive_kernel", rows)
    want = dict(nthr=nthr, gy=2 + 2 * k, smem=net_smem(par, k, nthr, adaptive=True))
    assert {key: f[key] for key in want} == want, (f, want)


def stats_of(ctx):
    s = ctx.network_stats()
    return numpy.array([s[name] for name in STATS], dtype=numpy.uint64)


def times_of(NT, T=2.0):
    return T * numpy.arange(1, NT + 1) / NT


def scales(k):
    from varsens_b200 import _cabi
    lo, hi = numpy.linspace(0.5, 1.0, k), numpy.linspace(1.5, 2.0, k)
    return ((_cabi.Scale(_cabi.SCALE_LINEAR, lo, hi), ("linear", lo, hi)),
            (_cabi.Scale(_cabi.SCALE_POWER, lo, hi), ("power", lo, hi)))


# (S, R, L, NT, k, nthr): l = L*NT from 1 to 64, the 64-thread form and the 32-thread form (64 trajectories of k + 8S + R
# doubles do not fit)
CASES = [
    pytest.param(1, 2, 1, 1, 3, 64, id="S1-l1-64thr"),
    pytest.param(6, 9, 4, 16, 5, 64, id="S6-l64-64thr"),
    pytest.param(12, 20, 3, 5, 8, 64, id="S12-l15-64thr"),
    pytest.param(64, 96, 2, 3, 12, 32, id="S64-l6-32thr"),
]


@pytest.mark.parametrize("S,R,L,NT,k,nthr", CASES)
def test_values_and_counts_equal_the_oracle(ctx, vb, monkeypatch, tmp_path, S, R, L, NT, k, nthr):
    """The whole design between NaN guards, a window starting mid-CTA, and raw (Sobol) points, values and all four step
    counts bit for bit; power scaling (device pow is not libm's) within 10 rtol."""
    trace = Tracer(ctx, monkeypatch, tmp_path)
    n = 8 * nthr + 37
    p = perm_of(n)
    rtol = 1e-7
    par = ob.adaptive_of(ob.random_network(5000 + S, S, R, L, k), times_of(NT), rtol=rtol, atol=1e-10)
    assert net_threads(par, k, adaptive=True) == nthr
    l = L * NT
    for sc, osc in ((None, None), scales(k)[0]):
        kw = {} if sc is None else dict(scale=sc)
        shape = (2 + 2 * k, n, l)
        got, lines = trace(lambda: guarded(ctx, shape, lambda out: ctx.eval_values(k, n, p, MAA, par, discard=3, out=out, **kw)))
        assert_form(lines, par, k, n, nthr)
        want, st = ob.values_adaptive(k, n, par, discard=3, scale=osc, perm=p)
        assert numpy.isfinite(want).all() and bits_equal(got, want), differ(got, want)
        assert (stats_of(ctx) == st).all(), (stats_of(ctx), st)
        i0, i1 = 37, n - 5
        win, lines = trace(lambda: ctx.eval_values(k, n, p, MAA, par, discard=3, i_begin=i0, i_end=i1, **kw))
        assert_form(lines, par, k, i1 - i0, nthr)
        want, st = ob.values_adaptive(k, n, par, discard=3, scale=osc, i0=i0, i1=i1, perm=p)
        assert bits_equal(win.reshape(want.shape), want) and bits_equal(win.reshape(want.shape), got[:, i0:i1])
        assert (stats_of(ctx) == st).all(), (stats_of(ctx), st)
    lin, olin = scales(k)[0]
    raw = vb.sobol_raw(k, n)
    got = ctx.eval_values(k, n, p, MAA, par, raw=raw, scale=lin)
    want, st = ob.values_adaptive(k, n, par, scale=olin, perm=p, raw=raw)
    assert bits_equal(got.reshape(want.shape), want) and (stats_of(ctx) == st).all()
    pw, opw = scales(k)[1]
    got = ctx.eval_values(k, n, p, MAA, par, scale=pw)
    want, _ = ob.values_adaptive(k, n, par, scale=opw, perm=p)
    numpy.testing.assert_allclose(got.reshape(want.shape), want, rtol=10 * rtol, atol=1e-9)


def test_fit_boundary_and_limits_launch_nothing(ctx, vb, monkeypatch, tmp_path):
    """A network of 104 species (at k = 6 the 32-thread form holds at most 111) with the most reactions that fit runs and
    matches the oracle;
    one more reaction is VS_ERR_UNSUPPORTED, VS_FLAG_SEPARABLE is VS_ERR_UNSUPPORTED and L*NT > 64 is VS_ERR_ARG, all before
    anything is launched."""
    from varsens_b200 import _cabi
    trace = Tracer(ctx, monkeypatch, tmp_path)
    S, L, NT, k, nthr = 104, 2, 2, 6, 32
    n = 8 * nthr + 37
    p = perm_of(n)
    full = ob.random_network(4343, S, 512, L, k)

    def first(R):
        net = ob.unpack(full, adaptive=False)
        net.rec = net.rec[:R]
        return ob.adaptive_of(ob.pack(net), [0.5, 1.0], rtol=1e-6, atol=1e-10)
    limit = optin()
    R = max(r for r in range(1, 512) if net_smem(first(r), k, nthr, adaptive=True) <= limit)
    assert R >= 16 and net_smem(first(R + 1), k, nthr, adaptive=True) > limit, R
    assert net_smem(first(R), k, 64, adaptive=True) > limit, R
    par = first(R)
    lin, olin = scales(k)[0]
    got, lines = trace(lambda: guarded(ctx, (2 + 2 * k, n, L * NT), lambda out: ctx.eval_values(k, n, p, MAA, par, scale=lin,
                                                                                                 out=out)))
    assert_form(lines, par, k, n, nthr)
    want, st = ob.values_adaptive(k, n, par, scale=olin, perm=p)
    assert numpy.isfinite(want).all() and bits_equal(got, want), differ(got, want)
    assert (stats_of(ctx) == st).all()
    before = ctx.launch_count()
    with pytest.raises(vb.VarsensError) as e:
        ctx.eval_values(k, n, p, MAA, first(R + 1), scale=lin)
    assert e.value.status == ERR_UNSUPPORTED
    with pytest.raises(vb.VarsensError) as e:
        ctx.run_fused(k, n, p, MAA, first(R + 1), scale=lin)
    assert e.value.status == ERR_UNSUPPORTED
    small = ob.adaptive_of(ob.chain_network(2), [1.0])
    with pytest.raises(vb.VarsensError) as e:
        ctx.run_fused(4, 16, perm_of(16), MAA, small, flags=_cabi.FLAG_SECOND_ORDER | _cabi.FLAG_SEPARABLE)
    assert e.value.status == ERR_UNSUPPORTED
    wide = ob.adaptive_of(ob.random_network(7, 4, 6, 5, 4), times_of(13))
    with pytest.raises(vb.VarsensError) as e:
        ctx.eval_values(4, 16, perm_of(16), MAA, wide)
    assert e.value.status == ERR_ARG
    assert ctx.launch_count() == before


def test_rejections_and_failures(ctx, vb):
    """A first step far too large makes every trajectory reject; a small max_steps gives NaN in exactly the oracle's positions
    and leaves every other value bit-identical to the unlimited run."""
    k, n = 4, 8 * 64 + 37
    p = perm_of(n)
    lin, olin = scales(k)[0]
    fixed = ob.random_network(606, 8, 12, 2, k)
    times = [0.5, 1.0, 2.0, 4.0]
    par = ob.adaptive_of(fixed, times, rtol=1e-9, atol=1e-12, h0=2.0)
    got = ctx.eval_values(k, n, p, MAA, par, scale=lin)
    want, st = ob.values_adaptive(k, n, par, scale=olin, perm=p)
    assert bits_equal(got, want) and (stats_of(ctx) == st).all()
    assert st[1] >= (2 + 2 * k) * n and st[2] == 0
    util = float(st[0] + st[1]) / float(st[3])
    assert 0.0 < util <= 1.0
    cap = int(0.75 * float(st[0] + st[1]) / ((2 + 2 * k) * n))               # below the mean attempts per trajectory
    capped = ob.adaptive_of(fixed, times, rtol=1e-9, atol=1e-12, h0=2.0, max_steps=cap)
    got2 = ctx.eval_values(k, n, p, MAA, capped, scale=lin)
    want2, st2 = ob.values_adaptive(k, n, capped, scale=olin, perm=p)
    nan = numpy.isnan(want2)
    assert nan.any() and (~nan).any() and st2[2] > 0
    assert bits_equal(got2, want2) and (stats_of(ctx) == st2).all()
    assert (numpy.isnan(got2) == nan).all() and bits_equal(got2[~nan], got[~nan])
    assert int(st2[2]) == int(numpy.isnan(want2[..., -1]).sum())


@pytest.mark.parametrize("L,NT", [(1, 1), (2, 3)])
def test_indices_through_the_two_phase_route(ctx, vb, L, NT):
    import torch
    from varsens_b200 import _cabi, dist
    k, n = 5, 600
    l = L * NT
    p = perm_of(n)
    par = ob.adaptive_of(ob.random_network(88 + L, 6, 9, L, k), times_of(NT), rtol=1e-8, atol=1e-12)
    sc = _cabi.Scale(_cabi.SCALE_LINEAR, numpy.full(k, 0.5), numpy.full(k, 2.0))
    vals, st = ob.values_adaptive(k, n, par, scale=("linear", 0.5, 2.0), perm=p)
    ref = oexact.indices(vals.reshape(-1, l), k, n)
    for flags in (0, _cabi.FLAG_SECOND_ORDER):
        res = ctx.run_fused(k, n, p, MAA, par, scale=sc, flags=flags)
        assert (stats_of(ctx) == st).all()
        for name in (NAMES if flags else NAMES[:6]):
            close(numpy.asarray(getattr(res, name)), ref[name].reshape(numpy.asarray(getattr(res, name)).shape))
    whole = ctx.run_fused(k, n, p, MAA, par, scale=sc)
    assert whole.sens.shape == (k, l) and whole.sens_2.shape == (k, l, k, l)
    plen = dist.partials_layout(k, l)["length"]
    parts = []
    for a, b in ((0, 97), (97, 350), (350, n)):
        parts.append(ctx.fused_partials(k, n, p, MAA, par, scale=sc, i_begin=a, i_end=b))
        _, sw = ob.values_adaptive(k, n, par, scale=("linear", 0.5, 2.0), perm=p, i0=a, i1=b)
        assert (stats_of(ctx) == sw).all(), (a, b)              # the shard's rows only, not base row 0 of the common shift
    summed = ctx.finalize(k, l, n, parts[0] + parts[1] + parts[2])
    for name in NAMES:
        close(getattr(summed, name), getattr(whole, name))
    peer = torch.zeros(2 * 1 * plen * 2 + 16, dtype=torch.float64, device="cuda")
    one = ctx.run_fused_p2p(k, n, p, MAA, par, 1, 0, [peer.data_ptr()], [peer.data_ptr()], 1, 0, n, scale=sc)
    for name in NAMES:
        assert bits_equal(getattr(one, name), getattr(whole, name)), name


def test_python_api(ctx, vb):
    k, n, NT = 4, 64, 3
    P = vb.Param
    args = (["A", "B", "C"],
            [(["A"], ["B"], P(0), P(1)), (["B", "B"], ["C"], P(2)), (["C"], [], 0.3), ([], ["A"], P(3))],
            [1.0, 0.2, 0.0], [{"A": 1.0}, {"B": 1.0, "C": 2.0}])
    net = vb.AdaptiveMassActionNetwork(*args, times=[0.5, 1.0, 2.0], rtol=1e-8, atol=1e-12)
    lo, hi = numpy.full(k, 0.5), numpy.full(k, 2.0)
    scaling = lambda x: vb.linear(x, lo, hi)                                # noqa: E731
    v = vb.Varsens(net, scaling, k, n, verbose=False)
    assert v.E_2.shape == (2 * NT,) and v.sens.shape == (k, 2 * NT) and v.sens_2.shape == (k, 2 * NT, k, 2 * NT)
    want, _ = ob.values_adaptive(k, n, net.params(k), scale=("linear", lo, hi))
    o = v.objective
    assert o.fM_1.shape == (n, 2 * NT) and o.fN_j.shape == (k, n, 2 * NT) and o.flat().shape == (2 * n * (1 + k), 2 * NT)
    assert bits_equal(o.fM_1, want[0]) and bits_equal(o.fN_j, want[2:2 + k])
    course = o.fM_1.reshape(n, NT, 2)                                       # the time course of observable 0 and 1
    assert bits_equal(course[:, 2, 1], want[0, :, 5])
    ref = oexact.indices(want.reshape(-1, 2 * NT), k, n)
    for name in NAMES:
        close(getattr(v, name), ref[name])
    short = vb.AdaptiveMassActionNetwork(*args, times=[0.5, 1.0, 2.0], rtol=1e-8, atol=1e-12, max_steps=6)
    with pytest.warns(RuntimeWarning, match=r"\d+ trajectories failed"):
        w = vb.Varsens(short, scaling, k, n, verbose=False)
    assert numpy.isnan(w.sens).any()
    with pytest.warns(RuntimeWarning, match=r"\d+ trajectories failed"):
        vals = vb.Objective(k, n, w.sample, short, verbose=False).flat()
    assert numpy.isnan(vals).any()
