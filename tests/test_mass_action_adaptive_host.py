"""CPU checks of the adaptive mass-action network objective (VS_OBJ_MASS_ACTION_ADAPTIVE): the host validation behind
vs_objective_outputs, the packed layout AdaptiveMassActionNetwork builds, and the oracle's frozen Dormand-Prince 5(4)
stepper against closed forms and scipy's DOP853 at tight tolerances."""
import ctypes
import math

import numpy
import pytest

from oracle import mass_action as ob


@pytest.fixture(scope="module")
def cabi():
    import __graft_entry__ as g
    g.build()
    from varsens_b200 import _cabi
    return _cabi


def outputs(cabi, k, params):
    par = numpy.ascontiguousarray(params, dtype=numpy.float64)
    l = ctypes.c_int(-7)
    st = cabi.lib().vs_objective_outputs(int(k), cabi.OBJ_MASS_ACTION_ADAPTIVE, par.ctypes.data_as(ctypes.c_void_p),
                                         int(par.size), ctypes.byref(l))
    return st, l.value


def ab_network(L=1, times=(0.5, 1.0), kr=None, rtol=1e-8, atol=1e-12):
    """A -> B (kf = 1) or A <-> B (kf = 1, kr), A(0) = 1; L observables of B."""
    rec = [0, -1, 1, -1, -1, 1.0, -1, 0.0 if kr is None else kr]
    return numpy.array([2, 1, L, len(times), rtol, atol, 1e-6, 100000] + rec + [-1, 1.0, -1, 0.0] + [0.0, 1.0] * L +
                       list(times), dtype=numpy.float64)


def test_outputs_are_l_times_nt(cabi):
    assert outputs(cabi, 1, ab_network()) == (0, 2)
    assert outputs(cabi, 1, ab_network(3, times=(1, 2, 3, 4))) == (0, 12)
    assert outputs(cabi, 1, ab_network(8, times=range(1, 9))) == (0, 64)            # L*NT = 64 is the limit
    assert outputs(cabi, 1, ab_network(64, times=(1.0,))) == (0, 64)
    assert outputs(cabi, 1, ab_network(5, times=range(1, 14)))[0] == 1              # 65
    assert outputs(cabi, 1, ab_network(1, times=range(1, 66)))[0] == 1              # 65
    assert outputs(cabi, 16, ob.adaptive_of(ob.random_network(3, 128, 192, 8, 16), [1.0, 2.0])) == (0, 16)
    # the fixed-step objective keeps its own header
    assert outputs(cabi, 1, ob.chain_network(1))[0] == 1
    st = ctypes.c_int()
    par = ob.chain_network(1)
    assert cabi.lib().vs_objective_outputs(2, cabi.OBJ_MASS_ACTION, par.ctypes.data_as(ctypes.c_void_p), int(par.size),
                                           ctypes.byref(st)) == 0 and st.value == 1


@pytest.mark.parametrize("field,value", [
    (3, 0),             # NT < 1
    (3, 1.5),           # NT not an integer
    (4, -1e-9),         # rtol < 0
    (4, math.inf),      # rtol not finite
    (4, math.nan),
    (5, 0.0),           # atol <= 0
    (5, -1.0),
    (5, math.inf),
    (6, 0.0),           # h0 <= 0
    (6, -1e-3),
    (6, math.nan),
    (7, 0),             # max_steps < 1
    (7, 2.5),           # max_steps not an integer
    (7, 2.0 ** 31),     # max_steps >= 2^31
    (7, math.inf),
    (8, 2),             # reactant species index == S (the limits of VS_OBJ_MASS_ACTION)
    (12, 1),            # kf coordinate == k
    (0, 129),           # S > 128
    (2, 0),             # L = 0
    (-2, 0.0),          # t_1 not > 0
    (-2, -0.5),
    (-1, 0.5),          # not strictly increasing (t_2 == t_1)
    (-1, 0.25),         # decreasing
    (-1, math.inf),     # not finite
    (-2, math.nan),
])
def test_malformed_adaptive_network_is_refused(cabi, field, value):
    p = ab_network()
    p[field] = value
    st, _ = outputs(cabi, 1, p)
    assert st == 1, cabi.lib().vs_last_error()


def test_adaptive_sizes_are_checked(cabi):
    p = ab_network()
    assert outputs(cabi, 1, p[:-1])[0] == 1                                         # one time short
    assert outputs(cabi, 1, numpy.append(p, 2.0))[0] == 1                           # NT says 2, three times follow
    assert outputs(cabi, 1, p[:7])[0] == 1                                          # header cut short
    assert outputs(cabi, 0, p)[0] == 1                                              # k out of range
    q = ab_network()
    q[3] = 3
    assert outputs(cabi, 1, numpy.append(q, 3.0))[0] == 0                           # NT = 3 with three times


def test_adaptive_object_builds_the_documented_layout(cabi):
    import varsens_b200 as vb
    P = vb.Param
    net = vb.AdaptiveMassActionNetwork(["A", "B", "C"],
                                       [(["A", "A"], "B", P(0), P(1)), ([], ["C"], 0.5), (["C"], [], 2),
                                        ([1, "C"], ["B", "C"], 1.25, 0.75)],
                                       [1.0, P(2), 0], [{"B": 2.0, "C": -1.0}, "A"], times=[0.5, 2.0, 3.0], rtol=1e-7,
                                       atol=1e-10, h0=1e-4, max_steps=500)
    want = [3, 4, 2, 3, 1e-7, 1e-10, 1e-4, 500,
            0, 0, 1, -1, 0, 0.0, 1, 0.0,
            -1, -1, 2, -1, -1, 0.5, -1, 0.0,
            2, -1, -1, -1, -1, 2.0, -1, 0.0,
            1, 2, 1, 2, -1, 1.25, -1, 0.75,
            -1, 1.0, 2, 0.0, -1, 0.0,
            0.0, 2.0, -1.0, 1.0, 0.0, 0.0,
            0.5, 2.0, 3.0]
    assert net.params(3).tolist() == want
    assert net.outputs(3) == 6
    with pytest.raises(vb.VarsensError, match="coordinate 2"):
        net.params(2)
    # the shared parsing leaves MassActionNetwork's packing as it was; h0 defaults to 1e-6 * times[-1]
    fixed = vb.MassActionNetwork(2, [([0], [1], 1.0)], [1.0, 0.0], [1], nsteps=3)
    assert fixed.params(1).tolist() == [2, 1, 1, 0.01, 3, 0, -1, 1, -1, -1, 1.0, -1, 0.0, -1, 1.0, -1, 0.0, 0.0, 1.0]
    d = vb.AdaptiveMassActionNetwork(2, [([0], [1], 1.0)], [1.0, 0.0], [1], times=[4.0])
    assert d.params(1).tolist() == [2, 1, 1, 1, 1e-6, 1e-9, 4e-6, 100000, 0, -1, 1, -1, -1, 1.0, -1, 0.0, -1, 1.0, -1, 0.0,
                                    0.0, 1.0, 4.0]
    assert numpy.array_equal(d.params(1), ob.adaptive_of(vb.MassActionNetwork(2, [([0], [1], 1.0)], [1.0, 0.0], [1]).params(1),
                                                           [4.0]))


@pytest.mark.parametrize("bad", [
    dict(times=[]),
    dict(times=[0.0, 1.0]),
    dict(times=[1.0, 1.0]),
    dict(times=[2.0, 1.0]),
    dict(times=[1.0, float("inf")]),
    dict(times=[[1.0, 2.0]]),
    dict(times="1.0"),
    dict(times=list(range(1, 66))),
    dict(observables=["A", "B"], times=list(range(1, 34))),
    dict(rtol=-1e-6),
    dict(rtol=float("nan")),
    dict(atol=0.0),
    dict(atol="1e-9"),
    dict(h0=0.0),
    dict(h0=-1.0),
    dict(max_steps=0),
    dict(max_steps=2 ** 31),
    dict(max_steps=10.0),
    dict(species=["A", "A"]),
    dict(reactions=[(["Z"], [], 1.0)]),
])
def test_adaptive_object_rejects_bad_input(cabi, bad):
    import varsens_b200 as vb
    args = dict(species=["A", "B"], reactions=[(["A"], ["B"], 1.0)], initial=[1.0, 0.0], observables=["B"], times=[1.0])
    args.update(bad)
    with pytest.raises(vb.VarsensError):
        vb.AdaptiveMassActionNetwork(**args)


TIMES = (0.1, 0.5, 1.0, 2.0, 3.5, 5.0)


def test_oracle_decay_matches_closed_form():
    v, info = ob.points_values([[0.0]], ab_network(2, TIMES))
    t = numpy.repeat(TIMES, 2)
    assert numpy.abs(v[0] - (1.0 - numpy.exp(-t))).max() < 1e-7
    assert info[0, 2] == 0 and info[0, 1] >= len(TIMES)


def test_oracle_reversible_pair_matches_closed_form():
    kf, kr = 1.0, 0.4
    v, info = ob.points_values([[0.0]], ab_network(1, TIMES, kr=kr))
    exact = kf / (kf + kr) * (1.0 - numpy.exp(-(kf + kr) * numpy.array(TIMES)))
    assert numpy.abs(v[0] - exact).max() < 1e-7 and info[0, 2] == 0


def _stiffish(seed, S, R, k):
    """A seeded network with one fast reversible pair X_0 <-> X_1 (rates 300 and 200) added to it."""
    net = ob.unpack(ob.random_network(seed, S, R, 2, k), adaptive=False)
    net.rec = numpy.vstack([net.rec, [0, -1, 1, -1, -1, 300.0, -1, 200.0]])
    return ob.pack(net)


NETS = [("random", 11, 4, 6, 3), ("random", 12, 9, 14, 5), ("random", 13, 12, 18, 6), ("stiffish", 14, 8, 10, 4)]


def _points(k, count, seed):
    return numpy.random.RandomState(seed).uniform(0.5, 2.0, size=(count, k))


@pytest.mark.parametrize("kind,seed,S,R,k", NETS)
def test_oracle_agrees_with_solve_ivp(kind, seed, S, R, k):
    fixed = ob.random_network(seed, S, R, 2, k) if kind == "random" else _stiffish(seed, S, R, k)
    times = [0.25, 1.0, 2.0]
    pts = _points(k, 3, seed)
    ref = numpy.array([ob.solve_ivp_values(ob.adaptive_of(fixed, times), x) for x in pts])
    errs = []
    for rtol in (1e-4, 1e-6, 1e-8):
        v, info = ob.points_values(pts, ob.adaptive_of(fixed, times, rtol=rtol, atol=1e-12))
        assert (info[:, 2] == 0).all()
        d = numpy.abs(v - ref)
        errs.append(d.max())
        if rtol == 1e-8:
            assert (d <= 1e-6 * numpy.abs(ref) + 1e-10).all(), d.max()
    assert errs[0] > errs[1] > errs[2], errs


def test_small_max_steps_gives_nan_from_the_failing_time():
    times = (0.5, 1.0, 2.0, 4.0)
    pts = _points(3, 64, 5)
    fixed = ob.random_network(21, 5, 8, 2, 3)
    full, info = ob.points_values(pts, ob.adaptive_of(fixed, times, rtol=1e-9, atol=1e-12))
    assert (info[:, 2] == 0).all()
    cap = int(numpy.median(info[:, 0]))
    v, capped = ob.points_values(pts, ob.adaptive_of(fixed, times, rtol=1e-9, atol=1e-12, max_steps=cap))
    failed = capped[:, 2] == 1
    assert failed.any() and (~failed).any()
    assert (capped[:, 0] <= cap).all() and (capped[failed, 0] == cap).all()
    for p in range(len(pts)):
        nan = numpy.isnan(v[p])
        if not failed[p]:
            assert not nan.any() and (v[p].view(numpy.int64) == full[p].view(numpy.int64)).all()
            continue
        first = int(numpy.argmax(nan))                      # NaN from the first unreached time on, the rest identical
        assert first % 2 == 0 and nan[first:].all() and not nan[:first].any()
        assert (v[p, :first].view(numpy.int64) == full[p, :first].view(numpy.int64)).all()
    k, n = 3, 8
    vals, stats = ob.values_adaptive(k, n, ob.adaptive_of(fixed, times, max_steps=3), scale=("linear", 0.5, 2.0))
    assert vals.shape == (2 + 2 * k, n, 2 * len(times))
    assert int(stats[2]) == int(numpy.isnan(vals[..., -1]).sum()) == (2 + 2 * k) * n
