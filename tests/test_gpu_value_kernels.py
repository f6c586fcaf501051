"""The point-by-point value kernels of the two-phase path past their first CTA, in every launch form, against the oracle.

eval_values_kernel (kernels_vals.cu) runs one thread per base row with the row's A_i and B_i in shared memory,
[coordinate][thread]: 128 threads up to k = 48 (the > 48 KB opt-in from k = 25), 64 threads for k = 49 ... 96, 32 threads
beyond.  The RK4 chain takes its heavy route (grid.y = 2 + 2k, one point per thread); Ishigami, and the g-function when the
product-form kernel declines (VS_NO_PF_EVAL=1, Horner mode), the light route (every point of a row in one thread).
network_values_kernel (kernels_network.cu) integrates one mass-action trajectory per thread, with the network tables and a
[variable][thread] state in shared memory: 64 threads, or 32 when 64 trajectories do not fit.

Every launch checked here has at least 8 CTAs and a ragged last one (n = 8 nthr + 37), and the VS_TRACE line of the launch
shows that the intended form ran.  A row index, block layout or shared-memory size that is right only in the first CTA shows.
  A. the RK4 chain bit for bit against cport.values (linear scaling is exact, so device and oracle integrate the same rates);
  B. the light route: the g-function at rtol 1e-13, Ishigami within a bound on its terms (the device sin is not libm's),
     and Horner mode's points where the Halton bases exceed 255;
  C. mass-action networks bit for bit against oracle.mass_action in both forms, every source and Halton arithmetic, the
     largest network the 32-thread form holds, and the edges of the description (nsteps = 0, dt < 0);
  D. network indices with three outputs through the two-phase route with the Gram kernel in steady state, and ragged shards
     with a host and a device permutation."""
import math

import numpy
import pytest

from conftest import close
from oracle import cport, exact as oexact, halton as ohalton, mass_action as ob, pipeline
from test_gpu_kernel_forms import TOP, disc, straddle
from test_gpu_mass_action import bits_equal
from test_gpu_steady_state import Tracer, assert_gram_steady, gparams, gram_lines, switches
from varsens_b200._cabi import OBJ_MASS_ACTION

pytestmark = pytest.mark.gpu

NAMES = ("E_2", "var_y", "U_j", "U_nj", "sens", "sens_t", "sens_2", "sens_2n")
GF, ISHI, RK4 = cport.OBJ_GFUNCTION, cport.OBJ_ISHIGAMI, cport.OBJ_RK4_CHAIN
MA = OBJ_MASS_ACTION
ERR_ARG, ERR_UNSUPPORTED = 1, 5
PAD = 64                                             # NaN guard elements on each side of a device output buffer
EPS = numpy.finfo(numpy.float64).eps


@pytest.fixture(scope="module")
def vb():
    import varsens_b200
    return varsens_b200


@pytest.fixture(scope="module")
def ctx(vb):
    return vb.Context.get(0)


def perm_of(n):
    return pipeline.permutation(n).astype(numpy.uint32)


def eval_threads(k):
    """Block size launch_eval_t picks: the largest of 128, 64, 32 whose A/B rows take <= 96 KB of shared memory."""
    nthr = 128
    while nthr > 32 and 2 * k * nthr * 8 > 96 * 1024:
        nthr //= 2
    return nthr


def launch_line(lines, name, rows):
    """The one trace line of kernel `name` with `rows` base rows; it has >= 8 CTAs and a ragged last one."""
    got = [f for nm, f in lines if nm == name and f["rows"] == rows]
    assert len(got) == 1, (name, rows, lines)
    f = got[0]
    assert f["gx"] == -(-rows // f["nthr"]) and f["gx"] >= 8 and rows % f["nthr"] != 0, (name, f)
    return f


def assert_eval_form(lines, k, rows, heavy):
    f = launch_line(lines, "eval_values_kernel", rows)
    nthr = eval_threads(k)
    want = dict(nthr=nthr, ppc=1 if heavy else 2 + 2 * k, gy=2 + 2 * k if heavy else 1, smem=2 * k * nthr * 8)
    assert {key: f[key] for key in want} == want, (k, heavy, f)
    assert not [x for x in lines if x[0] == "eval_values_pf_kernel"], lines
    return f


def guarded(ctx, shape, call):
    """call(out=...) into the middle of a NaN-filled device buffer; checks that exactly the output's doubles were written
    around it and returns them as a host array of `shape`."""
    import torch
    cnt = int(numpy.prod(shape))
    buf = torch.full((cnt + 2 * PAD,), float("nan"), dtype=torch.float64, device="cuda")
    call(out=buf[PAD:PAD + cnt])
    torch.cuda.synchronize()
    h = buf.cpu().numpy()
    assert numpy.isnan(h[:PAD]).all() and numpy.isnan(h[PAD + cnt:]).all(), "a write outside the output"
    return h[PAD:PAD + cnt].reshape(shape)


def differ(got, want):
    bad = numpy.flatnonzero(numpy.asarray(got).view(numpy.int64).ravel() != numpy.asarray(want).view(numpy.int64).ravel())
    return "%d of %d differ, first at %s" % (bad.size, numpy.asarray(want).size, bad[:8])


# ------------------------------------------------------------------------------------------------
# A. RK4 chain, heavy route
# ------------------------------------------------------------------------------------------------
# (k, nsteps) -> functor: RK4Chain<S> for k / 2 in 1..10, 12, 16; RK4ChainDyn otherwise (k / 2 <= 64 links).  A step moves
# mass at most four links on, so nsteps >= k / 8 keeps the last species' amount, the value, away from an exact 0.
RK4_CASES = (
    pytest.param(6, 60, id="k6-chain3-128thr"),
    pytest.param(32, 30, id="k32-chain16-128thr-optin"),
    pytest.param(40, 30, id="k40-dyn-128thr-optin"),
    pytest.param(60, 20, id="k60-dyn-64thr"),
    pytest.param(100, 15, id="k100-dyn-32thr"),
    pytest.param(128, 20, id="k128-dyn-32thr-64links"),
)


def _rk4_scale(k):
    from varsens_b200 import _cabi
    r = numpy.linspace(0.5, 2.0, k)
    return _cabi.Scale(_cabi.SCALE_LINEAR, r * 0.5, r * 2.0), ("linear", r * 0.5, r * 2.0)


@pytest.mark.parametrize("k,nsteps", RK4_CASES)
def test_rk4_chain_every_form(ctx, monkeypatch, tmp_path, k, nsteps):
    """The whole design into a NaN-guarded device buffer, a window starting mid-CTA, and a run at Halton index 2^32 - 1, each
    bit for bit against the oracle's trajectories."""
    trace = Tracer(ctx, monkeypatch, tmp_path)
    nthr = eval_threads(k)
    n = 8 * nthr + 37
    p = perm_of(n)
    par = [0.02, nsteps]
    sc, osc = _rk4_scale(k)
    shape = (2 + 2 * k, n)
    want = cport.values(k, n, RK4, par, discard=777, scale=osc)
    assert numpy.isfinite(want).all() and (want > 0).all()
    whole, lines = trace(lambda: guarded(ctx, shape, lambda out: ctx.eval_values(k, n, p, RK4, par, discard=777, scale=sc,
                                                                                    out=out)))
    assert bits_equal(whole, want), differ(whole, want)
    assert_eval_form(lines, k, n, heavy=True)
    lo, hi = 37, n - 5
    win, lines = trace(lambda: ctx.eval_values(k, n, p, RK4, par, discard=777, scale=sc, i_begin=lo, i_end=hi))
    assert_eval_form(lines, k, hi - lo, heavy=True)
    assert bits_equal(win, whole[:, lo:hi]), differ(win, whole[:, lo:hi])
    d = disc(k, n, TOP)
    top, lines = trace(lambda: ctx.eval_values(k, n, p, RK4, par, discard=d, scale=sc))
    assert_eval_form(lines, k, n, heavy=True)
    want = cport.values(k, n, RK4, par, discard=d, scale=osc)
    assert bits_equal(top, want), differ(top, want)


def test_rk4_chain_link_limit(ctx, vb):
    """64 links is the chain's limit (RK4ChainDyn's register arrays): k = 130 is refused before anything is launched."""
    k, n = 130, 64
    sc, _ = _rk4_scale(k)
    before = ctx.launch_count()
    with pytest.raises(vb.VarsensError) as e:
        ctx.eval_values(k, n, perm_of(n), RK4, [0.02, 10], scale=sc)
    assert e.value.status == ERR_ARG
    assert ctx.launch_count() == before


# ------------------------------------------------------------------------------------------------
# B. light route: g-function and Ishigami
# ------------------------------------------------------------------------------------------------
LIGHT_KS = (pytest.param(6, id="k6-128thr"), pytest.param(30, id="k30-128thr-optin"), pytest.param(70, id="k70-64thr"),
            pytest.param(130, id="k130-32thr"))


@pytest.mark.parametrize("k", LIGHT_KS)
def test_gfunction_point_by_point(ctx, monkeypatch, tmp_path, k):
    """The g-function where the product-form kernel declines: VS_NO_PF_EVAL=1 (whole design into a NaN-guarded device buffer,
    and a window starting mid-CTA) and Horner mode, whose points come from the oracle's restatement of that arithmetic.
    rtol 1e-13: the device's term is fma(|fma(4, x, -2)|, inv, off), a few ulp from the oracle's."""
    trace = Tracer(ctx, monkeypatch, tmp_path)
    n = 8 * eval_threads(k) + 37
    a, p = gparams(k), perm_of(n)
    want = cport.values(k, n, GF, a, discard=777)
    got, lines = trace(lambda: guarded(ctx, (2 + 2 * k, n), lambda out: ctx.eval_values(k, n, p, GF, a, discard=777, out=out)),
                       VS_NO_PF_EVAL=1)
    assert_eval_form(lines, k, n, heavy=False)
    numpy.testing.assert_allclose(got, want, rtol=1e-13, atol=0)
    lo, hi = 37, n - 5
    win, lines = trace(lambda: ctx.eval_values(k, n, p, GF, a, discard=777, i_begin=lo, i_end=hi), VS_NO_PF_EVAL=1)
    assert_eval_form(lines, k, hi - lo, heavy=False)
    assert bits_equal(win, got[:, lo:hi]), differ(win, got[:, lo:hi])

    def horner():
        ctx.set_halton_mode(3)
        return ctx.eval_values(k, n, p, GF, a)
    got, lines = trace(horner)
    assert_eval_form(lines, k, n, heavy=False)
    raw = ohalton.halton_points_mode(k, 20 * k + 1, 2 * n, "horner")
    numpy.testing.assert_allclose(got, cport.values(k, n, GF, a, raw=raw), rtol=1e-13, atol=0)


@pytest.mark.parametrize("k,n", ((55, 97), (70, 97), (453, 16)))
def test_horner_points_past_base_255(ctx, monkeypatch, k, n):
    """Horner mode's points bit for bit against the oracle's restatement where the bases no longer fit a byte: dimension 54
    has base 257, and k = 453 reaches base 3203.  The export kernel and the point-by-point kernels share the digit loop
    (radical_inverse_horner), which once kept the digits in 8 bits."""
    p = perm_of(n)
    for discard in (0, disc(k, n, TOP)):
        raw = ohalton.halton_points_mode(k, 20 * k + discard + 1, 2 * n, "horner")
        want = cport.sample_flat(k, n, perm=p, raw=raw)
        with switches(ctx, monkeypatch):
            ctx.set_halton_mode(3)
            got = ctx.sample_flat(k, n, p, discard)
        assert bits_equal(got, want), (discard, differ(got, want))


@pytest.mark.parametrize("k", (pytest.param(3, id="k3-128thr"),) + LIGHT_KS[1:])
def test_ishigami_every_form(ctx, monkeypatch, tmp_path, k):
    """Ishigami on [-pi, pi]^k (only x_0 .. x_2 enter) against the oracle: the device sin is not libm's, so the bound is on the
    terms, |got - want| <= 8 eps (|s0| + A s1^2 + B x2^4 |s0|), from the oracle's points."""
    from varsens_b200 import _cabi
    trace = Tracer(ctx, monkeypatch, tmp_path)
    n = 8 * eval_threads(k) + 37
    p = perm_of(n)
    A, B = 7.0, 0.1
    sc = _cabi.Scale(_cabi.SCALE_LINEAR, numpy.full(k, -math.pi), numpy.full(k, math.pi))
    osc = ("linear", [-math.pi] * k, [math.pi] * k)
    got, lines = trace(lambda: guarded(ctx, (2 + 2 * k, n), lambda out: ctx.eval_values(k, n, p, ISHI, [A, B], discard=99,
                                                                                          scale=sc, out=out)))
    assert_eval_form(lines, k, n, heavy=False)
    want = cport.values(k, n, ISHI, [A, B], discard=99, scale=osc)
    x = cport.sample_flat(k, n, 99, osc).reshape(2 + 2 * k, n, k)
    s0, s1, x2 = numpy.sin(x[..., 0]), numpy.sin(x[..., 1]), x[..., 2]
    bound = 8 * EPS * (numpy.abs(s0) + A * s1 * s1 + B * x2 ** 4 * numpy.abs(s0))
    err = numpy.abs(got - want)
    assert (err <= bound).all(), "max error / bound %.3g" % (err / bound).max()
    lo, hi = 37, n - 5
    win, lines = trace(lambda: ctx.eval_values(k, n, p, ISHI, [A, B], discard=99, scale=sc, i_begin=lo, i_end=hi))
    assert_eval_form(lines, k, hi - lo, heavy=False)
    assert bits_equal(win, got[:, lo:hi]), differ(win, got[:, lo:hi])


# ------------------------------------------------------------------------------------------------
# C. mass-action networks
# ------------------------------------------------------------------------------------------------
def net_smem(par, k, nthr, adaptive=False):
    """Shared memory of network_values_kernel: the tables (40 bytes a reaction, 4 per species pointer and list entry, rounded
    up to 16 bytes), then k + 3S + R doubles per trajectory.  network_adaptive_kernel: network_values_kernel's tables, the
    output times and observable lists (8 bytes a time and weight, 4 per observable pointer and species, rounded up to 16),
    then k + 8S + R doubles per trajectory."""
    net = ob.unpack(par, adaptive)
    up = lambda b: -(-b // 16) * 16                                 # noqa: E731
    table = up(40 * net.R + 4 * (net.S + 1 + net.nnz))
    if adaptive:
        return table + up(8 * (net.NT + net.nobs) + 4 * (net.L + 1 + net.nobs)) + (k + 8 * net.S + net.R) * nthr * 8
    return table + (k + 3 * net.S + net.R) * nthr * 8


def optin():
    import torch
    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


def net_threads(par, k, adaptive=False):
    return 64 if net_smem(par, k, 64, adaptive) <= optin() else 32


def assert_net_form(lines, par, k, rows, nthr):
    f = launch_line(lines, "network_values_kernel", rows)
    want = dict(nthr=nthr, gy=2 + 2 * k, smem=net_smem(par, k, nthr))
    assert {key: f[key] for key in want} == want, (f, want)
    return f


def _net_scales(k):
    from varsens_b200 import _cabi
    lo, hi = numpy.linspace(0.5, 1.0, k), numpy.linspace(1.5, 2.0, k)
    return (_cabi.Scale(_cabi.SCALE_LINEAR, lo, hi), ("linear", lo, hi)), (_cabi.Scale(_cabi.SCALE_POWER, lo, hi), ("power", lo, hi))


def _net_sources(vb, k, n):
    """(name, Halton mode, eval_values kwargs, oracle kwargs, exact): the oracle gets the points of a Halton mode as raw."""
    (lin, olin), (pw, opw) = _net_scales(k)
    sob = vb.sobol_raw(k, n)
    out = [("identity", 0, {}, {}, True),
           ("linear-discard", 0, dict(discard=777, scale=lin), dict(discard=777, scale=olin), True),
           ("power", 0, dict(scale=pw), dict(scale=opw), False),
           ("sobol-raw", 0, dict(raw=sob, scale=lin), dict(raw=sob, scale=olin), True)]
    for mode in (1, 2, 3):
        raw = ohalton.halton_points_mode(k, 20 * k + 5 + 1, 2 * n, ohalton.MODES[mode])
        out.append(("halton-mode%d" % mode, mode, dict(discard=5, scale=lin), dict(raw=raw, scale=olin), True))
    for name, d in (("L2^32-1", disc(k, n, TOP)), ("P37^6", straddle(k, n, 37 ** 6))):
        out.append((name, 0, dict(discard=d, scale=lin), dict(discard=d, scale=olin), True))
    return out


# (S, R, L, k, nthr, nsteps): the 64-thread form and the 32-thread form (64 trajectories of k + 3S + R doubles do not fit);
# few steps for the large network, whose oracle is slow
NET_FORMS = (pytest.param(12, 20, 8, 6, 64, 30, id="S12-R20-64thr"),
             pytest.param(128, 192, 8, 16, 32, 8, id="S128-R192-32thr"))


@pytest.mark.parametrize("S,R,L,k,nthr,nsteps", NET_FORMS)
def test_network_sources_and_modes(ctx, vb, monkeypatch, tmp_path, S, R, L, k, nthr, nsteps):
    """Identity, linear scaling with a discard, power scaling (rtol 1e-12: pow is <= 2 ulp), raw Sobol points, Halton modes
    1 - 3, the largest Halton index and a straddle of 37^6, each into a NaN-guarded device buffer and bit for bit against the
    oracle (power aside)."""
    trace = Tracer(ctx, monkeypatch, tmp_path)
    n = 8 * nthr + 37
    p = perm_of(n)
    par = ob.random_network(1000 + S, S, R, L, k, dt=0.01, nsteps=nsteps)
    assert net_threads(par, k) == nthr
    shape = (2 + 2 * k, n, L)
    for name, mode, kw, okw, exact in _net_sources(vb, k, n):
        def run():
            ctx.set_halton_mode(mode)
            return guarded(ctx, shape, lambda out: ctx.eval_values(k, n, p, MA, par, out=out, **kw))
        got, lines = trace(run)
        assert_net_form(lines, par, k, n, nthr)
        want = ob.values(k, n, par, perm=p, **okw)
        assert numpy.isfinite(want).all(), name
        if exact:
            assert bits_equal(got, want), (name, differ(got, want))
        else:
            numpy.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-300, err_msg=name)


@pytest.mark.parametrize("S,R,L,k,nthr,nsteps", NET_FORMS)
def test_network_windows_and_edges(ctx, vb, monkeypatch, tmp_path, S, R, L, k, nthr, nsteps):
    """Windows that start mid-CTA equal the slice of the whole run, host and device output alike; nsteps = 0 gives the
    observables of the initial amounts (some of them coordinates); dt < 0 integrates backwards, bit for bit with the oracle."""
    trace = Tracer(ctx, monkeypatch, tmp_path)
    n = 8 * nthr + 37
    p = perm_of(n)
    (lin, olin), _ = _net_scales(k)
    par = ob.random_network(2000 + S, S, R, L, k, dt=0.01, nsteps=nsteps)
    whole, lines = trace(lambda: ctx.eval_values(k, n, p, MA, par, discard=3, scale=lin))
    assert_net_form(lines, par, k, n, nthr)
    want = ob.values(k, n, par, discard=3, scale=olin, perm=p)
    assert bits_equal(whole, want), differ(whole, want)
    for lo, hi in ((37, n - 5), (nthr + 7, n)):
        win, lines = trace(lambda: ctx.eval_values(k, n, p, MA, par, discard=3, scale=lin, i_begin=lo, i_end=hi))
        assert_net_form(lines, par, k, hi - lo, nthr)
        assert bits_equal(win, whole[:, lo:hi]), (lo, hi, differ(win, whole[:, lo:hi]))
        dev = guarded(ctx, win.shape, lambda out: ctx.eval_values(k, n, p, MA, par, discard=3, scale=lin, i_begin=lo, i_end=hi,
                                                                  out=out))
        assert bits_equal(dev, win), (lo, hi, differ(dev, win))
    # nsteps = 0: the weighted sums of the initial amounts
    net = ob.unpack(par, adaptive=False)
    net.head["nsteps"] = 0
    par0 = ob.pack(net)
    init = net.init
    assert (init[:, 0] >= 0).any() and (init[:, 0] < 0).any()
    got, lines = trace(lambda: ctx.eval_values(k, n, p, MA, par0, discard=3, scale=lin))
    assert_net_form(lines, par0, k, n, nthr)
    want = ob.values(k, n, par0, discard=3, scale=olin, perm=p)
    assert bits_equal(got, want), differ(got, want)
    x = cport.sample_flat(k, n, 3, olin, perm=p)
    X0 = numpy.where(init[:, 0] >= 0, x[:, numpy.maximum(init[:, 0], 0).astype(int)], init[:, 1])
    err = numpy.abs(got.reshape(-1, L) - X0 @ net.w.T)
    assert (err <= 4 * S * EPS * (numpy.abs(X0) @ numpy.abs(net.w).T)).all()
    # dt < 0 (short: backwards, second-order reactions blow up in finite time)
    parn = ob.random_network(3000 + S, S, R, L, k, dt=-0.002, nsteps=10)
    got, lines = trace(lambda: ctx.eval_values(k, n, p, MA, parn, scale=lin))
    assert_net_form(lines, parn, k, n, nthr)
    want = ob.values(k, n, parn, scale=olin, perm=p)
    assert numpy.isfinite(want).all() and bits_equal(got, want), differ(got, want)


def test_network_fit_boundary(ctx, vb, monkeypatch, tmp_path):
    """The largest network the 32-thread form holds (S = 128, k = 16: one more reaction would not fit the device's opt-in
    shared memory) runs and matches the oracle bit for bit; with that one more reaction it is refused with
    VS_ERR_UNSUPPORTED before anything is launched."""
    trace = Tracer(ctx, monkeypatch, tmp_path)
    S, L, k, nthr = 128, 2, 16, 32
    n = 8 * nthr + 37
    p = perm_of(n)
    full = ob.random_network(4242, S, 512, L, k, dt=0.01, nsteps=4)

    def first(R):
        """The network of the first R reactions of `full` (same initial amounts and observables)."""
        net = ob.unpack(full, adaptive=False)
        net.rec = net.rec[:R]
        return ob.pack(net)
    limit = optin()
    R = max(r for r in range(1, 512) if net_smem(first(r), k, nthr) <= limit)
    assert R < 511 and net_smem(first(R + 1), k, nthr) > limit and net_smem(first(R), k, 64) > limit, R
    par = first(R)
    (lin, olin), _ = _net_scales(k)
    got, lines = trace(lambda: guarded(ctx, (2 + 2 * k, n, L), lambda out: ctx.eval_values(k, n, p, MA, par, scale=lin,
                                                                                             out=out)))
    assert_net_form(lines, par, k, n, nthr)
    want = ob.values(k, n, par, scale=olin, perm=p)
    assert numpy.isfinite(want).all() and bits_equal(got, want), differ(got, want)
    before = ctx.launch_count()
    with pytest.raises(vb.VarsensError) as e:
        ctx.eval_values(k, n, p, MA, first(R + 1), scale=lin)
    assert e.value.status == ERR_UNSUPPORTED
    assert ctx.launch_count() == before


# ------------------------------------------------------------------------------------------------
# D. network indices through the two-phase route, Gram kernel in steady state
# ------------------------------------------------------------------------------------------------
def test_network_indices_steady_state(ctx, vb, monkeypatch, tmp_path):
    """run_fused with three outputs at second order: values to HBM by network_values_kernel, then the general-form Gram
    kernel with every CTA past its stage ring three times.  The values are the oracle's bit for bit on the first, a middle and
    the ragged last CTA; the indices are the extended-precision estimators of those values.  Three ragged shards (two with
    i_begin != 0, whose shared shift f(M_1[0]) is a separate one-row launch) add up to the whole and finalize to the same
    indices, with a host permutation (row 0's entry staged on its own) and with a device one (read through the tensor)."""
    import torch
    trace = Tracer(ctx, monkeypatch, tmp_path)
    k, L, nthr = 5, 3, 64
    n = (1 << 18) + (1 << 16) + 7
    p = perm_of(n)
    par = ob.random_network(80, 6, 9, L, k, nsteps=40)
    (lin, olin), _ = _net_scales(k)
    res, lines = trace(lambda: ctx.run_fused(k, n, p, MA, par, scale=lin))
    assert_net_form(lines, par, k, n, nthr)
    g = gram_lines(lines)
    assert len(g) == 1, lines
    assert_gram_steady(g[0])
    vals = ctx.eval_values(k, n, p, MA, par, scale=lin)
    last = (n // nthr) * nthr
    for lo, hi in ((0, nthr), ((n // nthr // 2) * nthr, (n // nthr // 2 + 1) * nthr), (last, n)):
        want = ob.values(k, n, par, scale=olin, i0=lo, i1=hi, perm=p)
        assert bits_equal(vals[:, lo:hi], want), (lo, hi, differ(vals[:, lo:hi], want))
    ref = oexact.indices(vals.reshape(-1, L), k, n)
    for name in NAMES:
        close(numpy.asarray(getattr(res, name)), ref[name].reshape(numpy.asarray(getattr(res, name)).shape))
    whole = ctx.fused_partials(k, n, p, MA, par, scale=lin)
    shards = ((0, 100003), (100003, 100004), (100004, n))
    parts = {}
    for perm_name, perm in (("host", p), ("device", torch.from_numpy(p.astype(numpy.int32)).cuda())):
        acc = numpy.zeros_like(whole)
        for lo, hi in shards:
            part, lines = trace(lambda: ctx.fused_partials(k, n, perm, MA, par, scale=lin, i_begin=lo, i_end=hi))
            assert [f["rows"] for nm, f in lines if nm == "network_values_kernel"] == [hi - lo] + ([1] if lo else []), lines
            parts[perm_name, lo] = part
            acc += part
        numpy.testing.assert_allclose(acc, whole, rtol=1e-12, atol=1e-9, err_msg=perm_name)
        summed = ctx.finalize(k, L, n, acc)
        for name in NAMES:
            close(getattr(summed, name), ref[name].reshape(numpy.asarray(getattr(summed, name)).shape))
    for lo, hi in shards:
        assert bits_equal(parts["device", lo], parts["host", lo]), lo
