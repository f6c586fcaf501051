"""CPU checks of the result block on the Python side (_cabi.Result): the views of a flat buffer, the unpacked copy of one,
a fresh Result and its vs_result struct all follow the library's order E_2 var_y U_j U_nj sens sens_t sens_2 sens_2n."""
import ctypes

import numpy
import pytest

from varsens_b200 import _cabi

FIELDS = ("E_2", "var_y", "U_j", "U_nj", "sens", "sens_t", "sens_2", "sens_2n")
CASES = [(k, l, second) for k in (1, 6, 20) for l in (1, 3) for second in (True, False)]


def expected(k, l, flat, second_order):
    """The fields of a result block, written out independently of _cabi; None for sens_2 / sens_2n of a first-order block."""
    kl = k * l
    sizes = (l, l, kl, kl, kl, kl, kl * kl, kl * kl)
    shapes = ((l,), (l,), (k, l), (k, l), (k, l), (k, l), (k, l, k, l), (k, l, k, l))
    out, at = {}, 0
    for name, cnt, shape in zip(FIELDS, sizes, shapes):
        if name.startswith("sens_2") and not second_order:
            out[name] = None
            continue
        out[name] = flat[at:at + cnt].reshape(shape)
        at += cnt
    return out, at


@pytest.mark.parametrize("k,l,second_order", CASES)
def test_views_and_from_flat_agree(k, l, second_order):
    n = _cabi.Result.flat_len(k, l)
    assert n == 2 * l + 4 * k * l + 2 * (k * l) ** 2
    flat = numpy.arange(n, dtype=numpy.float64) + 0.5                    # every element distinct
    want, used = expected(k, l, flat, second_order)
    assert used == (n if second_order else 2 * l + 4 * k * l)
    v = _cabi.Result.views(k, l, flat, second_order)
    u = _cabi.Result.from_flat(k, l, flat, second_order)
    assert (v.k, v.l) == (u.k, u.l) == (k, l)
    for name in FIELDS:
        a, b, w = getattr(v, name), getattr(u, name), want[name]
        if w is None:
            assert a is None and b is None, name
            continue
        assert a.shape == b.shape == w.shape, name
        assert a.dtype == b.dtype == numpy.float64, name
        assert (a == w).all() and (b == w).all(), name
        assert numpy.shares_memory(a, flat) and not numpy.shares_memory(b, flat), name


@pytest.mark.parametrize("k,l,second_order", CASES)
def test_fresh_result_and_c_struct(k, l, second_order):
    r = _cabi.Result(k, l, second_order)
    cs = r.c_struct()
    for name in FIELDS:
        a = getattr(r, name)
        ptr = getattr(cs, name)
        if name.startswith("sens_2") and not second_order:
            assert a is None and ptr is None, name
            continue
        shape = (l,) if name in ("E_2", "var_y") else (k, l) if not name.startswith("sens_2") else (k, l, k, l)
        assert a.shape == shape and a.dtype == numpy.float64 and (a == 0).all(), name
        assert ptr == a.ctypes.data, name
    assert ctypes.sizeof(cs) == len(FIELDS) * ctypes.sizeof(ctypes.c_void_p)
