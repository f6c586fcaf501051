"""CPU checks of the stiff mass-action network objective (VS_OBJ_MASS_ACTION_STIFF): the host validation behind
vs_objective_outputs (exactly that of VS_OBJ_MASS_ACTION_ADAPTIVE), the Python ``method=`` keyword, the oracle's sparse factor
sizes, and the oracle's frozen Rodas3 stepper against scipy's Radau at tight tolerances on a stiff network."""
import ctypes

import numpy
import pytest

from oracle import mass_action as ob, mass_action_stiff as ost
import test_mass_action_adaptive_host as adaptive_host
from test_mass_action_adaptive_host import ab_network

# the adaptive host test's malformed descriptions (field, value)
MALFORMED = [m for m in adaptive_host.test_malformed_adaptive_network_is_refused.pytestmark if m.name == "parametrize"][0].args[1]


@pytest.fixture(scope="module")
def cabi():
    import __graft_entry__ as g
    g.build()
    from varsens_b200 import _cabi
    return _cabi


def outputs(cabi, k, params, objective):
    par = numpy.ascontiguousarray(params, dtype=numpy.float64)
    l = ctypes.c_int(-7)
    st = cabi.lib().vs_objective_outputs(int(k), int(objective), par.ctypes.data_as(ctypes.c_void_p), int(par.size),
                                         ctypes.byref(l))
    return st, l.value


def both(cabi, k, params):
    """(status, l) of the stiff objective, checked equal to the adaptive objective's."""
    a = outputs(cabi, k, params, cabi.OBJ_MASS_ACTION_ADAPTIVE)
    s = outputs(cabi, k, params, cabi.OBJ_MASS_ACTION_STIFF)
    assert s[0] == a[0] and (s[0] != 0 or s[1] == a[1]), (s, a)
    return s


def test_stiff_outputs_are_those_of_the_adaptive_objective(cabi):
    assert both(cabi, 1, ab_network()) == (0, 2)
    assert both(cabi, 1, ab_network(3, times=(1, 2, 3, 4))) == (0, 12)
    assert both(cabi, 1, ab_network(8, times=range(1, 9))) == (0, 64)
    assert both(cabi, 1, ab_network(5, times=range(1, 14)))[0] == 1                 # L*NT = 65
    assert both(cabi, 16, ob.adaptive_of(ob.random_network(3, 128, 192, 8, 16), [1.0, 2.0])) == (0, 16)
    p = ab_network()
    assert both(cabi, 1, p[:-1])[0] == 1 and both(cabi, 1, numpy.append(p, 2.0))[0] == 1 and both(cabi, 0, p)[0] == 1
    assert both(cabi, 2, ob.chain_network(1))[0] == 1                                # a fixed-step header is not a stiff one


@pytest.mark.parametrize("field,value", MALFORMED)
def test_malformed_stiff_network_is_refused(cabi, field, value):
    p = ab_network()
    p[field] = value
    assert both(cabi, 1, p)[0] == 1, cabi.lib().vs_last_error()


def test_method_keyword(cabi):
    import varsens_b200 as vb
    args = (["A", "B"], [(["A"], ["B"], 1.0, 0.5)], [1.0, 0.0], ["B"])
    default = vb.AdaptiveMassActionNetwork(*args, times=[1.0, 2.0])
    stiff = vb.AdaptiveMassActionNetwork(*args, times=[1.0, 2.0], method="rodas3")
    assert default.objective_id == cabi.OBJ_MASS_ACTION_ADAPTIVE == 4 and default.method == "dopri5"
    assert vb.AdaptiveMassActionNetwork(*args, times=[1.0, 2.0], method="dopri5").objective_id == 4
    assert stiff.objective_id == cabi.OBJ_MASS_ACTION_STIFF == 5 and stiff.method == "rodas3"
    assert numpy.array_equal(stiff.params(1), default.params(1)) and stiff.outputs(1) == 2
    for bad in ("radau", "RODAS3", "", None, 5):
        with pytest.raises(vb.VarsensError, match="method"):
            vb.AdaptiveMassActionNetwork(*args, times=[1.0], method=bad)


def fast_pair(kf, kr):
    """tools/bench_mass_action_adaptive.py's fast pair: seeded network 7 (S=8, R=12, L=2, k=8) plus X_0 <-> X_1 at kf, kr."""
    net = ob.unpack(ob.random_network(7, 8, 12, 2, 8, dt=0.01, nsteps=1000), adaptive=False)
    net.rec = numpy.vstack([net.rec, [0, -1, 1, -1, -1, kf, -1, kr]])
    return ob.pack(net)


@pytest.mark.parametrize("fixed,nlu", [
    (ob.chain_network(10), 31),
    (fast_pair(1e3, 8e2), 25),
    (ob.random_network(2024, 32, 48, 4, 64), 221),
    (ob.random_network(3, 128, 192, 8, 16), 1552),
])
def test_factor_sizes(fixed, nlu):
    """Nonzeros of L+U under minimum-degree order (the natural order gives 31, 29, 343 and 4037, dense S^2 121 .. 16384)."""
    sz = ost.stiff_sizes(ob.adaptive_of(fixed, [1.0]))
    assert sz["nlu"] == nlu and sz["nlu"] == sz["nlow"] + sz["nup"] + ob.unpack(fixed, False).S
    assert sorted(sz["ord"].tolist()) == list(range(ob.unpack(fixed, False).S))


def radau_values(params, x):
    from scipy.integrate import solve_ivp
    net = ob.unpack(params, True)
    f, y0 = ob.numpy_rhs(params, x)
    sol = solve_ivp(f, (0.0, net.times[-1]), y0, method="Radau", t_eval=net.times, rtol=1e-12, atol=1e-14)
    assert sol.success, sol.message
    return (net.w @ sol.y).T.reshape(net.NT * net.L)


PTS = numpy.random.RandomState(3).uniform(0.5, 2.0, size=(2, 8))


def test_oracle_agrees_with_radau_on_the_fast_pair():
    fixed = fast_pair(1e3, 8e2)
    times = [0.5, 10.0]
    ref = numpy.array([radau_values(ob.adaptive_of(fixed, times), x) for x in PTS])
    errs = []
    for rtol, atol in ((1e-6, 1e-9), (1e-9, 1e-12)):
        v, info = ost.points_values(PTS, ob.adaptive_of(fixed, times, rtol=rtol, atol=atol))
        assert (info[:, 2] == 0).all() and numpy.isfinite(v).all()
        errs.append(numpy.abs(v - ref).max())
        if rtol == 1e-6:
            assert errs[0] <= 1e-6 and (info[:, 1] < 600).all(), (errs, info)
    assert errs[1] < errs[0] / 10, errs


def test_stiff_oracle_finishes_where_dopri5_fails():
    """Pair rates 1e5 / 8e4: Rodas3 needs a few hundred steps, Dormand-Prince exhausts max_steps = 100000 (NaN outputs)."""
    par = ob.adaptive_of(fast_pair(1e5, 8e4), [10.0], rtol=1e-6, atol=1e-9)
    v, info = ost.points_values(PTS[:1], par)
    assert info[0, 2] == 0 and info[0, 1] < 1000 and numpy.isfinite(v).all(), info
    assert numpy.abs(v[0] - radau_values(par, PTS[0])).max() <= 1e-6
    d, dinfo = ob.points_values(PTS[:1], par)
    assert dinfo[0, 2] == 1 and dinfo[0, 0] == 100000 and numpy.isnan(d).all(), dinfo


def test_small_max_steps_gives_nan_from_the_failing_time():
    times = (0.5, 1.0, 2.0, 4.0)
    pts = numpy.random.RandomState(5).uniform(0.5, 2.0, size=(48, 3))
    fixed = ob.random_network(21, 5, 8, 2, 3)
    full, info = ost.points_values(pts, ob.adaptive_of(fixed, times, rtol=1e-9, atol=1e-12))
    assert (info[:, 2] == 0).all()
    cap = int(numpy.median(info[:, 0]))
    v, capped = ost.points_values(pts, ob.adaptive_of(fixed, times, rtol=1e-9, atol=1e-12, max_steps=cap))
    failed = capped[:, 2] == 1
    assert failed.any() and (~failed).any() and (capped[failed, 0] == cap).all()
    for p in range(len(pts)):
        nan = numpy.isnan(v[p])
        first = int(numpy.argmax(nan)) if failed[p] else nan.size
        assert not nan[:first].any() and nan[first:].all() and first % 2 == 0
        assert (v[p, :first].view(numpy.int64) == full[p, :first].view(numpy.int64)).all()
