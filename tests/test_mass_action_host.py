"""CPU checks of the mass-action network objective: the host validation behind vs_objective_outputs, the packed layout
MassActionNetwork builds, and the oracle's frozen arithmetic (chain written as a network, closed-form A -> B)."""
import ctypes
import math

import numpy
import pytest

from oracle import cport, mass_action as ob


@pytest.fixture(scope="module")
def cabi():
    import __graft_entry__ as g
    g.build()
    from varsens_b200 import _cabi
    return _cabi


def outputs(cabi, k, objective, params):
    par = numpy.ascontiguousarray(params, dtype=numpy.float64)
    l = ctypes.c_int(-7)
    st = cabi.lib().vs_objective_outputs(int(k), int(objective), par.ctypes.data_as(ctypes.c_void_p), int(par.size),
                                         ctypes.byref(l))
    return st, l.value


def ab_network(L=1):
    # A -> B irreversible, kf = 1; L observables of B
    return numpy.array([2, 1, L, 0.01, 100] + [0, -1, 1, -1, -1, 1.0, -1, 0.0] + [-1, 1.0, -1, 0.0] + [0.0, 1.0] * L)


def test_outputs_of_existing_objectives(cabi):
    assert outputs(cabi, 6, cabi.OBJ_GFUNCTION, [0, 0.5, 3, 9, 99, 99]) == (0, 1)
    assert outputs(cabi, 3, cabi.OBJ_ISHIGAMI, [7.0, 0.1]) == (0, 1)
    assert outputs(cabi, 20, cabi.OBJ_RK4_CHAIN, [0.01, 1000]) == (0, 1)
    assert outputs(cabi, 2, cabi.OBJ_ISHIGAMI, [7.0, 0.1])[0] == 1           # same validation as the evaluating calls
    assert outputs(cabi, 5, cabi.OBJ_RK4_CHAIN, [0.01, 1000])[0] == 1
    assert outputs(cabi, 6, 9, [0.0])[0] == 1


def test_outputs_of_networks(cabi):
    assert outputs(cabi, 1, cabi.OBJ_MASS_ACTION, ab_network()) == (0, 1)
    assert outputs(cabi, 1, cabi.OBJ_MASS_ACTION, ab_network(3)) == (0, 3)
    assert outputs(cabi, 1, cabi.OBJ_MASS_ACTION, ab_network(64)) == (0, 64)
    assert outputs(cabi, 20, cabi.OBJ_MASS_ACTION, ob.chain_network(10)) == (0, 1)
    assert outputs(cabi, 16, cabi.OBJ_MASS_ACTION, ob.random_network(3, 128, 192, 8, 16)) == (0, 8)
    assert outputs(cabi, 4, cabi.OBJ_MASS_ACTION, ab_network()[:5])[0] == 1             # header only


@pytest.mark.parametrize("field,value", [
    (5, 2),          # reactant species index == S
    (7, 5),          # product species index > S
    (5, -2),         # species index below -1
    (9, 1),          # kf coordinate == k (k = 1)
    (11, 3),         # kr coordinate >= k
    (13, 1),         # initial-amount coordinate >= k
    (5, 0.5),        # non-integer species index
    (9, 0.25),       # non-integer coordinate
    (0, 129),        # S > 128
    (1, 513),        # R > 512
    (4, -1),         # negative nsteps
    (4, 2.0 ** 31),  # nsteps >= 2^31
    (4, 1.5),        # non-integer nsteps
    (3, math.inf),   # dt not finite
    (3, math.nan),
])
def test_malformed_network_is_refused(cabi, field, value):
    p = ab_network()
    p[field] = value
    st, _ = outputs(cabi, 1, cabi.OBJ_MASS_ACTION, p)
    assert st == 1, cabi.lib().vs_last_error()


def test_network_size_fields_are_checked(cabi):
    p = ab_network()
    assert outputs(cabi, 1, cabi.OBJ_MASS_ACTION, p[:-1])[0] == 1                     # wrong n_params
    assert outputs(cabi, 1, cabi.OBJ_MASS_ACTION, numpy.append(p, 0.0))[0] == 1
    q = ab_network(65)
    assert outputs(cabi, 1, cabi.OBJ_MASS_ACTION, q)[0] == 1                           # L > 64
    q = ab_network()
    q[2] = 0
    assert outputs(cabi, 1, cabi.OBJ_MASS_ACTION, q[:-2])[0] == 1                      # L = 0
    assert outputs(cabi, 1, cabi.OBJ_MASS_ACTION, p[:3])[0] == 1                       # header cut short
    assert outputs(cabi, 0, cabi.OBJ_MASS_ACTION, p)[0] == 1                           # k out of range


def test_network_object_builds_the_documented_layout(cabi):
    import varsens_b200 as vb
    P = vb.Param
    net = vb.MassActionNetwork(["A", "B", "C"],
                               [(["A", "A"], "B", P(0), P(1)),       # homodimer, reversible with a coordinate
                                ([], ["C"], 0.5),                    # synthesis
                                (["C"], [], 2),                      # degradation; an int rate is a constant
                                ([1, "C"], ["B", "C"], 1.25, 0.75)], # catalyst C, species by index
                               [1.0, P(2), 0],
                               [{"B": 2.0, "C": -1.0}, "A"], dt=0.02, nsteps=7)
    want = [3, 4, 2, 0.02, 7,
            0, 0, 1, -1, 0, 0.0, 1, 0.0,
            -1, -1, 2, -1, -1, 0.5, -1, 0.0,
            2, -1, -1, -1, -1, 2.0, -1, 0.0,
            1, 2, 1, 2, -1, 1.25, -1, 0.75,
            -1, 1.0, 2, 0.0, -1, 0.0,
            0.0, 2.0, -1.0, 1.0, 0.0, 0.0]
    assert net.params(3).tolist() == want
    assert net.outputs(3) == 2 and vb.RK4Chain().outputs(20) == 1
    with pytest.raises(vb.VarsensError, match="coordinate 2"):
        net.params(2)
    n2 = vb.MassActionNetwork(2, [([0], [1], 1.0)], [1.0, 0.0], [1], nsteps=3)
    assert n2.params(1).tolist() == [2, 1, 1, 0.01, 3, 0, -1, 1, -1, -1, 1.0, -1, 0.0, -1, 1.0, -1, 0.0, 0.0, 1.0]


@pytest.mark.parametrize("bad", [
    dict(species=0),
    dict(species=["A", "A"]),
    dict(reactions=[(["A", "B", "A"], [], 1.0)]),
    dict(reactions=[(["Z"], [], 1.0)]),
    dict(reactions=[([2], [], 1.0)]),
    dict(reactions=[(["A"], [], "1.0")]),
    dict(reactions=[(["A"], [], True)]),
    dict(reactions=[(["A"],)]),
    dict(reactions=[]),
    dict(initial=[1.0]),
    dict(observables=[]),
    dict(observables=[{"A": "x"}]),
    dict(observables=[True]),
    dict(nsteps=-1),
    dict(nsteps=2.5),
    dict(dt=float("inf")),
])
def test_network_object_rejects_bad_input(cabi, bad):
    import varsens_b200 as vb
    args = dict(species=["A", "B"], reactions=[(["A"], ["B"], 1.0)], initial=[1.0, 0.0], observables=["B"])
    args.update(bad)
    with pytest.raises(vb.VarsensError):
        vb.MassActionNetwork(**args)
    with pytest.raises(vb.VarsensError):
        vb.Param(-1)
    with pytest.raises(vb.VarsensError):
        vb.Param(1.0)


@pytest.mark.parametrize("k", range(2, 42, 2))
def test_oracle_chain_as_network_is_bit_identical(k):
    n = 6
    r = numpy.linspace(0.5, 2.0, k)
    sc = ("linear", r * 0.5, r * 2)
    chain = cport.values(k, n, cport.OBJ_RK4_CHAIN, [0.02, 60], scale=sc)
    net = ob.values(k, n, ob.chain_network(k // 2, 0.02, 60), scale=sc)
    assert net.shape == (2 + 2 * k, n, 1)
    assert (net[..., 0].view(numpy.int64) == chain.view(numpy.int64)).all()


def test_oracle_irreversible_decay_matches_closed_form():
    v = ob.values(1, 4, ab_network(2))
    assert v.shape == (4, 4, 2)
    exact = 1.0 - math.exp(-1.0)                       # B(T), T = 100 * 0.01
    assert numpy.abs(v - exact).max() < 1e-9           # RK4 global error ~ T * dt^4 / 120


def test_numpy_twin_is_close_to_the_oracle():
    k, n = 6, 16
    p = ob.random_network(5, 12, 18, 3, k, nsteps=40)
    v = ob.values(k, n, p, scale=("linear", 0.5, 2.0))
    flat = cport.sample_flat(k, n, scale=("linear", 0.5, 2.0))
    tw = ob.mass_action_rows(flat, p).reshape(2 + 2 * k, n, 3)
    numpy.testing.assert_allclose(tw, v, rtol=1e-12, atol=1e-13)
