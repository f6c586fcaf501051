"""GPU checks of the stiff mass-action network objective (VS_OBJ_MASS_ACTION_STIFF, network_rosenbrock_kernel): values and
step counts bit for bit against the oracle's Rodas3 restatement (oracle/mass_action_stiff.c: f_mass_action_stiff) in the 64- and
32-thread forms, past the first CTA; failures; the fit limit; indices through the two-phase route and ragged shards; the
Python API; agreement with the Dormand-Prince kernel on a non-stiff network.

Every launch checked against its VS_TRACE line has at least 8 CTAs and a ragged last one (n = 8 nthr + 37)."""
import numpy
import pytest

from conftest import close
from oracle import exact as oexact, mass_action as ob, mass_action_stiff as ost
from test_gpu_mass_action import bits_equal, perm_of
from test_gpu_steady_state import Tracer
from test_gpu_value_kernels import differ, guarded, launch_line, optin
from varsens_b200._cabi import OBJ_MASS_ACTION_ADAPTIVE, OBJ_MASS_ACTION_STIFF

pytestmark = pytest.mark.gpu

NAMES = ("E_2", "var_y", "U_j", "U_nj", "sens", "sens_t", "sens_2", "sens_2n")
MAS = OBJ_MASS_ACTION_STIFF
ERR_ARG, ERR_UNSUPPORTED = 1, 5
STATS = ("accepted", "rejected", "failed", "lane_work")


@pytest.fixture(scope="module")
def vb():
    import varsens_b200
    return varsens_b200


@pytest.fixture(scope="module")
def ctx(vb):
    return vb.Context.get(0)


def stiff_smem(par, k, nthr):
    """Shared memory of network_rosenbrock_kernel: network_adaptive_kernel's tables (40 bytes a reaction, 4 per species
    pointer and list entry; 8 a time and weight, 4 per observable pointer and species; each part rounded up to 16 bytes), the
    stiff tables (4 bytes each: jptr R+1, jcol and jtp 2 ncol + 1, jt, ord and piv 2S, lptr and uptr 2S + 2, the L and U
    entries, the update targets; rounded up to 16), then k + 7S + R + nnz(LU) doubles per trajectory."""
    net = ob.unpack(par, True)
    sz = ost.stiff_sizes(par)
    up = lambda b: -(-b // 16) * 16                                 # noqa: E731
    table = up(40 * net.R + 4 * (net.S + 1 + net.nnz)) + up(8 * (net.NT + net.nobs) + 4 * (net.L + 1 + net.nobs))
    table += up(4 * (4 * net.S + net.R + 4 + 2 * sz["ncol"] + sz["njt"] + sz["nlow"] + sz["nup"] + sz["nupd"]))
    return table + (k + 7 * net.S + net.R + sz["nlu"]) * nthr * 8


def stiff_threads(par, k):
    return 64 if stiff_smem(par, k, 64) <= optin() else 32


def assert_form(lines, par, k, rows, nthr):
    f = launch_line(lines, "network_rosenbrock_kernel", rows)
    want = dict(nthr=nthr, gy=2 + 2 * k, smem=stiff_smem(par, k, nthr))
    assert {key: f[key] for key in want} == want, (f, want)


def stats_of(ctx):
    s = ctx.network_stats()
    return numpy.array([s[name] for name in STATS], dtype=numpy.uint64)


def scales(k):
    from varsens_b200 import _cabi
    lo, hi = numpy.linspace(0.5, 1.0, k), numpy.linspace(1.5, 2.0, k)
    return ((_cabi.Scale(_cabi.SCALE_LINEAR, lo, hi), ("linear", lo, hi)),
            (_cabi.Scale(_cabi.SCALE_POWER, lo, hi), ("power", lo, hi)))


def with_pair(fixed, kf, kr):
    """The fixed-step description with a fast reversible pair X_0 <-> X_1 (rates kf, kr) appended: a stiff network."""
    net = ob.unpack(fixed, adaptive=False)
    net.rec = numpy.vstack([net.rec, [0, -1, 1, -1, -1, kf, -1, kr]])
    return ob.pack(net)


def features(par):
    """Which reaction kinds and table shapes the description exercises."""
    net = ob.unpack(par, True)
    rec = net.rec
    sides = [[int(s) for s in q[a:a + 2] if s >= 0] for q in rec for a in (0, 2)]
    sz = ost.stiff_sizes(par)
    P = numpy.eye(net.S, dtype=bool)                                 # the species pattern, for the fill
    N = net.N
    for r, q in enumerate(rec):
        rev = not (q[6] < 0 and q[7] == 0.0)
        cols = [int(s) for s in (list(q[0:2]) + (list(q[2:4]) if rev else [])) if s >= 0]
        for s in numpy.flatnonzero(N[:, r]):
            P[s, cols] = True
    perm = sz["ord"]
    return dict(homodimer=any(len(s) == 2 and s[0] == s[1] for s in sides),
                catalyst=any(set(int(s) for s in q[0:2] if s >= 0) & set(int(s) for s in q[2:4] if s >= 0) for q in rec),
                synthesis=any(not [s for s in q[0:2] if s >= 0] for q in rec),
                irreversible=any(q[6] < 0 and q[7] == 0.0 for q in rec),
                param_initial=bool((net.init[:, 0] >= 0).any()),
                fill=sz["nlu"] > int(P[numpy.ix_(perm, perm)].sum()))


# (seed, S, R, L, NT, k, pair, nthr): the 64-thread form and the 32-thread form (64 trajectories of k + 7S + R + nnz(LU)
# doubles do not fit); pair = rates of an appended fast reversible pair, or None
CASES = [
    pytest.param(6100, 6, 9, 2, 3, 5, (1e4, 8e3), 64, id="S6-l6-pair-64thr"),
    pytest.param(6200, 12, 20, 3, 5, 8, None, 64, id="S12-l15-64thr"),
    pytest.param(6300, 20, 32, 4, 16, 6, (1e5, 8e4), 64, id="S20-l64-pair-64thr"),
    pytest.param(6400, 40, 64, 2, 2, 12, (1e3, 8e2), 32, id="S40-l4-pair-32thr"),
]


@pytest.mark.parametrize("seed,S,R,L,NT,k,pair,nthr", CASES)
def test_values_and_counts_equal_the_oracle(ctx, vb, monkeypatch, tmp_path, seed, S, R, L, NT, k, pair, nthr):
    """The whole design between NaN guards, a window starting mid-CTA, and raw (Sobol) points, values and all four step
    counts bit for bit; power scaling (device pow is not libm's) within 10 rtol."""
    trace = Tracer(ctx, monkeypatch, tmp_path)
    n = 8 * nthr + 37
    p = perm_of(n)
    rtol = 1e-6
    fixed = ob.random_network(seed, S, R, L, k)
    par = ob.adaptive_of(fixed if pair is None else with_pair(fixed, *pair), 2.0 * numpy.arange(1, NT + 1) / NT, rtol=rtol,
                         atol=1e-10)
    assert stiff_threads(par, k) == nthr
    l = L * NT
    for sc, osc in ((None, None), scales(k)[0]):
        kw = {} if sc is None else dict(scale=sc)
        got, lines = trace(lambda: guarded(ctx, (2 + 2 * k, n, l), lambda out: ctx.eval_values(k, n, p, MAS, par, discard=3,
                                                                                                 out=out, **kw)))
        assert_form(lines, par, k, n, nthr)
        want, st = ost.values(k, n, par, discard=3, scale=osc, perm=p)
        assert numpy.isfinite(want).all() and bits_equal(got, want), differ(got, want)
        assert (stats_of(ctx) == st).all(), (stats_of(ctx), st)
        i0, i1 = 37, n - 5
        win, lines = trace(lambda: ctx.eval_values(k, n, p, MAS, par, discard=3, i_begin=i0, i_end=i1, **kw))
        assert_form(lines, par, k, i1 - i0, nthr)
        want, st = ost.values(k, n, par, discard=3, scale=osc, i0=i0, i1=i1, perm=p)
        assert bits_equal(win.reshape(want.shape), want) and bits_equal(win.reshape(want.shape), got[:, i0:i1])
        assert (stats_of(ctx) == st).all(), (stats_of(ctx), st)
    lin, olin = scales(k)[0]
    raw = vb.sobol_raw(k, n)
    got = ctx.eval_values(k, n, p, MAS, par, raw=raw, scale=lin)
    want, st = ost.values(k, n, par, scale=olin, perm=p, raw=raw)
    assert bits_equal(got.reshape(want.shape), want) and (stats_of(ctx) == st).all()
    pw, opw = scales(k)[1]
    got = ctx.eval_values(k, n, p, MAS, par, scale=pw)
    want, _ = ost.values(k, n, par, scale=opw, perm=p)
    numpy.testing.assert_allclose(got.reshape(want.shape), want, rtol=10 * rtol, atol=1e-9)


def test_cases_cover_the_reaction_kinds():
    """Together the networks of CASES have homodimers, catalysts, zero-order synthesis, irreversible reactions, initial
    amounts that are coordinates, and a factor with fill."""
    seen = {}
    for c in CASES:
        seed, S, R, L, NT, k, pair, _ = c.values
        fixed = ob.random_network(seed, S, R, L, k)
        for key, v in features(ob.adaptive_of(fixed if pair is None else with_pair(fixed, *pair), [1.0])).items():
            seen[key] = seen.get(key, False) or v
    assert all(seen.values()), seen


def test_failures_and_the_python_warning(ctx, vb):
    """A small max_steps gives NaN in exactly the oracle's positions, from the unreached time on, the oracle's failed count,
    and every other value bit-identical to the unlimited run; through the Python API it warns."""
    k, n = 4, 8 * 64 + 37
    p = perm_of(n)
    lin, olin = scales(k)[0]
    fixed = with_pair(ob.random_network(606, 8, 12, 2, k), 1e4, 8e3)
    times = [0.5, 1.0, 2.0, 4.0]
    par = ob.adaptive_of(fixed, times, rtol=1e-9, atol=1e-12)
    got = ctx.eval_values(k, n, p, MAS, par, scale=lin)
    want, st = ost.values(k, n, par, scale=olin, perm=p)
    assert bits_equal(got, want) and (stats_of(ctx) == st).all() and st[2] == 0
    assert 0.0 < float(st[0] + st[1]) / float(st[3]) <= 1.0
    cap = int(0.75 * float(st[0] + st[1]) / ((2 + 2 * k) * n))               # below the mean attempts per trajectory
    capped = ob.adaptive_of(fixed, times, rtol=1e-9, atol=1e-12, max_steps=cap)
    got2 = ctx.eval_values(k, n, p, MAS, capped, scale=lin)
    want2, st2 = ost.values(k, n, capped, scale=olin, perm=p)
    nan = numpy.isnan(want2)
    assert nan.any() and (~nan).any() and st2[2] > 0
    assert bits_equal(got2, want2) and (stats_of(ctx) == st2).all()
    assert (numpy.isnan(got2) == nan).all() and bits_equal(got2[~nan], got[~nan])
    assert int(st2[2]) == int(numpy.isnan(want2[..., -1]).sum())
    P = vb.Param
    args = (["A", "B", "C"], [(["A"], ["B"], P(0), P(1)), (["B", "B"], ["C"], P(2)), (["C"], [], 0.3), ([], ["A"], P(3))],
            [1.0, 0.2, 0.0], [{"A": 1.0}, {"B": 1.0, "C": 2.0}])
    short = vb.AdaptiveMassActionNetwork(*args, times=[0.5, 1.0, 2.0], rtol=1e-8, atol=1e-12, max_steps=4, method="rodas3")
    scaling = lambda x: vb.linear(x, numpy.full(k, 0.5), numpy.full(k, 2.0))  # noqa: E731
    with pytest.warns(RuntimeWarning, match=r"\d+ trajectories failed"):
        w = vb.Varsens(short, scaling, k, 64, verbose=False)
    assert numpy.isnan(w.sens).any()


def test_a_network_that_does_not_fit_launches_nothing(ctx, vb):
    """A network whose 32 trajectories do not fit is VS_ERR_UNSUPPORTED and names nnz(LU); VS_FLAG_SEPARABLE is
    VS_ERR_UNSUPPORTED; both before anything is launched."""
    from varsens_b200 import _cabi
    k = 16
    big = ob.adaptive_of(ob.random_network(3, 128, 192, 8, k), [1.0, 2.0])
    assert stiff_smem(big, k, 32) > optin()
    before = ctx.launch_count()
    for call in (lambda: ctx.eval_values(k, 64, perm_of(64), MAS, big), lambda: ctx.run_fused(k, 64, perm_of(64), MAS, big)):
        with pytest.raises(vb.VarsensError, match="nnz\\(LU\\) = 1552") as e:
            call()
        assert e.value.status == ERR_UNSUPPORTED
    small = ob.adaptive_of(ob.chain_network(2), [1.0])
    with pytest.raises(vb.VarsensError) as e:
        ctx.run_fused(4, 16, perm_of(16), MAS, small, flags=_cabi.FLAG_SECOND_ORDER | _cabi.FLAG_SEPARABLE)
    assert e.value.status == ERR_UNSUPPORTED
    assert ctx.launch_count() == before


def test_indices_and_ragged_shards(ctx, vb):
    """Varsens with method="rodas3" gives all eight indices within 1e-10 relative / 1e-12 absolute of the extended-precision
    oracle; ragged evaluation windows give the bits of one launch, ragged partial-sum shards add up to the whole, and the
    single-rank peer form gives its bits."""
    import torch
    from varsens_b200 import dist
    k, n, NT = 4, 600, 3
    P = vb.Param
    args = (["A", "B", "C", "D"],
            [(["A"], ["B"], P(0), P(1)), (["B", "B"], ["C"], P(2)), (["C"], [], 0.3), ([], ["A"], P(3)),
             (["A", "D"], ["C", "D"], 2.0, 0.5), (["C"], ["D"], 2e3, 1e3)],
            [1.0, 0.2, 0.0, P(3)], [{"A": 1.0}, {"B": 1.0, "D": 2.0}])
    net = vb.AdaptiveMassActionNetwork(*args, times=[0.5, 1.0, 2.0], rtol=1e-8, atol=1e-12, method="rodas3")
    lo, hi = numpy.full(k, 0.5), numpy.full(k, 2.0)
    v = vb.Varsens(net, lambda x: vb.linear(x, lo, hi), k, n, verbose=False)
    l = 2 * NT
    par = net.params(k)
    want, st = ost.values(k, n, par, scale=("linear", lo, hi))
    o = v.objective
    assert o.fM_1.shape == (n, l) and bits_equal(o.fM_1, want[0]) and bits_equal(o.fN_j, want[2:2 + k])
    ref = oexact.indices(want.reshape(-1, l), k, n)
    for name in NAMES:
        close(getattr(v, name), ref[name])
    p = perm_of(n)
    sc = vb._cabi.Scale(vb._cabi.SCALE_LINEAR, lo, hi)
    one = ctx.eval_values(k, n, p, MAS, par, scale=sc).reshape(2 + 2 * k, n, l)
    cuts = ((0, 97), (97, 350), (350, n))
    shards = [ctx.eval_values(k, n, p, MAS, par, scale=sc, i_begin=a, i_end=b).reshape(2 + 2 * k, b - a, l) for a, b in cuts]
    assert bits_equal(numpy.concatenate(shards, axis=1), one)
    whole = ctx.run_fused(k, n, p, MAS, par, scale=sc)
    assert (stats_of(ctx) == ost.values(k, n, par, scale=("linear", lo, hi), perm=p)[1]).all()
    parts = []
    for a, b in cuts:
        parts.append(ctx.fused_partials(k, n, p, MAS, par, scale=sc, i_begin=a, i_end=b))
        _, sw = ost.values(k, n, par, scale=("linear", lo, hi), perm=p, i0=a, i1=b)
        assert (stats_of(ctx) == sw).all(), (a, b)
    summed = ctx.finalize(k, l, n, parts[0] + parts[1] + parts[2])
    for name in NAMES:
        close(getattr(summed, name), getattr(whole, name))
    plen = dist.partials_layout(k, l)["length"]
    peer = torch.zeros(2 * 1 * plen * 2 + 16, dtype=torch.float64, device="cuda")
    single = ctx.run_fused_p2p(k, n, p, MAS, par, 1, 0, [peer.data_ptr()], [peer.data_ptr()], 1, 0, n, scale=sc)
    for name in NAMES:
        assert bits_equal(getattr(single, name), getattr(whole, name)), name


def test_agrees_with_dopri5_on_a_non_stiff_network(ctx):
    """Two different methods at rtol 1e-8, atol 1e-11: values agree to a tolerance-sized bound."""
    k, n = 6, 8 * 64 + 37
    p = perm_of(n)
    lin, _ = scales(k)[0]
    par = ob.adaptive_of(ob.random_network(77, 10, 16, 3, k), [0.5, 1.0, 2.0], rtol=1e-8, atol=1e-11)
    a = ctx.eval_values(k, n, p, OBJ_MASS_ACTION_ADAPTIVE, par, scale=lin)
    s = ctx.eval_values(k, n, p, MAS, par, scale=lin)
    assert numpy.isfinite(a).all() and numpy.isfinite(s).all()
    numpy.testing.assert_allclose(s, a, rtol=1e-6, atol=1e-8)
