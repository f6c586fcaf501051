"""GPU checks of the mass-action network objective (VS_OBJ_MASS_ACTION): the kernel against the RK4 chain and the oracle,
bit for bit where the scaling is exact; l > 1 outputs through the estimator entry points and the Python API; the limits."""
import numpy
import pytest

from conftest import close
from oracle import cport, exact as oexact, mass_action as ob, pipeline
from varsens_b200._cabi import OBJ_MASS_ACTION

pytestmark = pytest.mark.gpu

NAMES = ("E_2", "var_y", "U_j", "U_nj", "sens", "sens_t", "sens_2", "sens_2n")
MA, RK4 = OBJ_MASS_ACTION, cport.OBJ_RK4_CHAIN


@pytest.fixture(scope="module")
def vb():
    import varsens_b200
    return varsens_b200


@pytest.fixture(scope="module")
def ctx(vb):
    return vb.Context.get(0)


def perm_of(n):
    return pipeline.permutation(n).astype(numpy.uint32)


def bits_equal(a, b):
    a, b = numpy.ascontiguousarray(a, dtype=numpy.float64), numpy.ascontiguousarray(b, dtype=numpy.float64)
    return a.shape == b.shape and (a.view(numpy.int64) == b.view(numpy.int64)).all()


@pytest.mark.parametrize("k", [2, 4, 6, 8, 10, 12, 14, 16, 18, 20, 24, 32, 22])   # RK4Chain<S> for S <= 10, 12, 16; 22: RK4ChainDyn
def test_chain_as_network_equals_rk4_chain(ctx, vb, k):
    from varsens_b200 import _cabi
    n, discard = 40, 7
    r = numpy.linspace(0.5, 2.0, k)
    sc = _cabi.Scale(_cabi.SCALE_LINEAR, r * 0.5, r * 2.0)
    p = perm_of(n)
    chain = ctx.eval_values(k, n, p, RK4, [0.02, 120], discard=discard, scale=sc)
    net = ctx.eval_values(k, n, p, MA, ob.chain_network(k // 2, 0.02, 120), discard=discard, scale=sc)
    assert bits_equal(net, chain), "%d of %d values differ" % (int((net != chain).sum()), chain.size)
    if k in (4, 22):
        a = ctx.run_fused(k, n, p, RK4, [0.02, 120], discard=discard, scale=sc)
        b = ctx.run_fused(k, n, p, MA, ob.chain_network(k // 2, 0.02, 120), discard=discard, scale=sc)
        for name in NAMES:
            assert bits_equal(getattr(b, name), getattr(a, name)), name


NETS = [(1, 2, 1, 3), (3, 5, 3, 4), (12, 20, 8, 6), (40, 60, 3, 10), (128, 192, 8, 16)]   # S, R, L, k


@pytest.mark.parametrize("S,R,L,k", NETS)
def test_random_networks_equal_the_oracle(ctx, vb, S, R, L, k):
    import torch
    from varsens_b200 import _cabi
    n = 48
    p = perm_of(n)
    par = ob.random_network(1000 + S, S, R, L, k, dt=0.01, nsteps=60)
    lo, hi = numpy.linspace(0.5, 1.0, k), numpy.linspace(1.5, 2.0, k)
    for scale, osc in ((_cabi.IDENTITY, None), (_cabi.Scale(_cabi.SCALE_LINEAR, lo, hi), ("linear", lo, hi))):
        want = ob.values(k, n, par, discard=3, scale=osc, perm=p)
        got = ctx.eval_values(k, n, p, MA, par, discard=3, scale=scale)
        shape = (2 + 2 * k, n) + ((L,) if L > 1 else ())
        assert got.shape == shape and bits_equal(got, want.reshape(shape))
        assert numpy.isfinite(got).all()
        i0, i1 = 5, 31                                              # a window is the slice of the whole run
        win = ctx.eval_values(k, n, p, MA, par, discard=3, scale=scale, i_begin=i0, i_end=i1)
        assert bits_equal(win, got[:, i0:i1])
        # device output between NaN guards: exactly rows*(2+2k)*l doubles are written
        G, cnt = 64, (i1 - i0) * (2 + 2 * k) * L
        buf = torch.full((cnt + 2 * G,), float("nan"), dtype=torch.float64, device="cuda")
        ctx.eval_values(k, n, p, MA, par, discard=3, scale=scale, i_begin=i0, i_end=i1, out=buf[G:G + cnt])
        torch.cuda.synchronize()
        h = buf.cpu().numpy()
        assert numpy.isnan(h[:G]).all() and numpy.isnan(h[G + cnt:]).all()
        assert bits_equal(h[G:G + cnt], win.reshape(-1))
    sc = _cabi.Scale(_cabi.SCALE_POWER, lo, hi)
    got = ctx.eval_values(k, n, p, MA, par, scale=sc)
    want = ob.values(k, n, par, scale=("power", lo, hi), perm=p)
    numpy.testing.assert_allclose(got, want.reshape(got.shape), rtol=1e-12, atol=1e-300)


@pytest.mark.parametrize("L", [1, 3])
def test_indices_of_networks(ctx, vb, L):
    import torch
    from varsens_b200 import _cabi, dist
    k, n = 5, 600
    p = perm_of(n)
    par = ob.random_network(77 + L, 6, 9, L, k, nsteps=40)
    sc = _cabi.Scale(_cabi.SCALE_LINEAR, numpy.full(k, 0.5), numpy.full(k, 2.0))
    vals = ob.values(k, n, par, scale=("linear", 0.5, 2.0), perm=p).reshape(-1, L)
    ref = oexact.indices(vals, k, n)
    for flags in (0, _cabi.FLAG_SECOND_ORDER):
        res = ctx.run_fused(k, n, p, MA, par, scale=sc, flags=flags)
        names = NAMES if flags else NAMES[:6]
        for name in names:
            close(numpy.asarray(getattr(res, name)), ref[name].reshape(numpy.asarray(getattr(res, name)).shape))
    whole = ctx.run_fused(k, n, p, MA, par, scale=sc)
    assert whole.sens.shape == (k, L) and whole.sens_2.shape == (k, L, k, L)
    # three ragged shards of the partial sums add up to the whole
    plen = dist.partials_layout(k, L)["length"]
    parts = [ctx.fused_partials(k, n, p, MA, par, scale=sc, i_begin=a, i_end=b) for a, b in ((0, 97), (97, 350), (350, n))]
    assert all(x.shape == (plen,) for x in parts)
    summed = ctx.finalize(k, L, n, parts[0] + parts[1] + parts[2])
    for name in NAMES:
        close(getattr(summed, name), getattr(whole, name))
    # the one-call peer-memory form with a single rank equals vs_run_fused bit for bit
    peer = torch.zeros(2 * 1 * plen * 2 + 16, dtype=torch.float64, device="cuda")
    one = ctx.run_fused_p2p(k, n, p, MA, par, 1, 0, [peer.data_ptr()], [peer.data_ptr()], 1, 0, n, scale=sc)
    for name in NAMES:
        assert bits_equal(getattr(one, name), getattr(whole, name)), name
    assert dist.outputs_of_partials(k, plen) == L


def test_python_api(ctx, vb):
    k, n = 4, 64
    P = vb.Param
    net = vb.MassActionNetwork(["A", "B", "C"],
                               [(["A"], ["B"], P(0), P(1)), (["B", "B"], ["C"], P(2)), (["C"], [], 0.3), ([], ["A"], P(3))],
                               [1.0, 0.2, 0.0], [{"A": 1.0}, {"B": 1.0, "C": 2.0}], dt=0.02, nsteps=50)
    lo, hi = numpy.full(k, 0.5), numpy.full(k, 2.0)
    scaling = lambda x: vb.linear(x, lo, hi)                                # noqa: E731
    v = vb.Varsens(net, scaling, k, n, verbose=False)
    assert v.E_2.shape == (2,) and v.sens.shape == (k, 2) and v.sens_2.shape == (k, 2, k, 2)
    want = ob.values(k, n, net.params(k), scale=("linear", lo, hi))
    o = v.objective
    assert o.fM_1.shape == (n, 2) and o.fN_j.shape == (k, n, 2) and o.flat().shape == (2 * n * (1 + k), 2)
    assert bits_equal(o.fM_1, want[0]) and bits_equal(o.fN_j, want[2:2 + k])
    ref = oexact.indices(want.reshape(-1, 2), k, n)
    for name in NAMES:
        close(getattr(v, name), ref[name])
    # the numpy twin as a plain per-row callable (the reference's route)
    par = net.params(k)
    w = vb.Varsens(lambda x: ob.mass_action_row(x, par), scaling, k, n, verbose=False)
    for name in NAMES:
        close(getattr(w, name), getattr(v, name))


def test_limits_launch_nothing(ctx, vb):
    from varsens_b200 import _cabi
    k, n = 453, 4
    big = ob.random_network(9, 128, 512, 1, k)                 # k + 3S + R doubles per trajectory: 32 do not fit
    before = ctx.launch_count()
    with pytest.raises(vb.VarsensError) as e:
        ctx.eval_values(k, n, perm_of(n), MA, big)
    assert e.value.status == 5
    with pytest.raises(vb.VarsensError) as e:
        ctx.run_fused(k, n, perm_of(n), MA, big)
    assert e.value.status == 5
    with pytest.raises(vb.VarsensError) as e:
        ctx.run_fused(4, 16, perm_of(16), MA, ob.chain_network(2), flags=_cabi.FLAG_SECOND_ORDER | _cabi.FLAG_SEPARABLE)
    assert e.value.status == 5
    assert ctx.launch_count() == before
