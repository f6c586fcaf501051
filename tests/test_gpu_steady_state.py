"""The two-phase path -- estimators on given values and product-form evaluation -- in steady state.

Those kernels are persistent: a CTA of the Gram kernels loops over chunks of rows (the tensor-path gram_mma_kernel through a
ring of shared-memory stages, the register-tile gram_kernel through one staging buffer), a CTA of eval_values_pf_kernel over
32-row (NR = 1) or 64-row (NR = 2) tiles.  Every run here is long enough that each CTA takes several chunks or tiles, so the
ring wraps (stage parity flips, the producer waits on `empty` barriers the consumers really arrived on), the accumulators
carry over chunks, the last chunk is ragged in a CTA that already did full ones, and the next tile's permutation entry is
prefetched.  The trace lines of VS_TRACE name the form that ran and give its chunk or tile count per CTA; every case checks
them: chunks per CTA >= 3 x ring depth for the tensor path, >= 3 for the register-tile kernel, tiles per CTA >= 4.
  A. Gram kernels bit for bit on integer data (every summation order is exact), every form the host can pick, both modes.
  B. The contract tolerance at the size DESIGN.md §4.3 times (k = 20, n = 2^22), and with NaN-trimmed rows.
  C. Product-form values in steady state, and the two-phase route of run_fused / fused_partials at k > 20."""
import numpy
import pytest

from conftest import close
from oracle import cport, exact as oexact, pipeline

pytestmark = pytest.mark.gpu

A20 = [0, 0.5, 3, 9, 99, 99] + [99.0] * 14
NAMES = ("E_2", "var_y", "U_j", "U_nj", "sens", "sens_t", "sens_2", "sens_2n")
GF = cport.OBJ_GFUNCTION
SO = 1                                               # FLAG_SECOND_ORDER
PAD = 64                                             # NaN guard elements on each side of a device buffer (16-byte multiple)


@pytest.fixture(scope="module")
def ctx():
    import varsens_b200
    return varsens_b200.Context.get(0)


def perm_of(n):
    return pipeline.permutation(n).astype(numpy.uint32)


def gparams(k):
    return (A20 + [1.0, 2.0, 5.0, 99.0] * 30)[:k]


class switches(object):
    """VS_* switches for the body of a with-block (None = leave unset); afterwards every switch is back at its default."""

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


class Tracer(object):
    """Runs calls under VS_TRACE and returns the launch lines they appended: [(kernel, {key: int})]."""

    def __init__(self, ctx, monkeypatch, tmp_path):
        self.ctx, self.mp, self.path = ctx, monkeypatch, tmp_path / "trace.txt"

    def __call__(self, call, **env):
        if self.path.exists():
            self.path.unlink()
        with switches(self.ctx, self.mp, VS_TRACE=str(self.path), **env):
            out = call()
        lines = []
        if self.path.exists():
            for line in self.path.read_text().splitlines():
                words = line.split()
                if line.startswith("# ") and len(words) > 2 and all("=" in w for w in words[2:]):
                    lines.append((words[1], {w.split("=")[0]: int(w.split("=")[1]) for w in words[2:]}))
        return out, lines


def form(line):
    """The instantiation a trace line names: ("mma", ST, multi, guard, gen) or ("reg", T)."""
    name, f = line
    if name == "gram_mma_kernel":
        return ("mma", f["ST"], f["multi"], f["guard"], f["gen"])
    assert name == "gram_kernel", line
    return ("reg", f["T"])


def per_cta(items, grid):
    return -(-items // grid)


def assert_gram_steady(line):
    """Each CTA takes at least three rounds of the stage ring (tensor path) or three chunks (register-tile kernel)."""
    name, f = line
    if name == "gram_mma_kernel":
        chunks = per_cta(per_cta(f["rows"], f["rc"]), f["gx"])
        assert chunks >= 3 * f["nstage"], ("not in steady state", line, chunks)
    else:
        chunks = per_cta(per_cta(f["rows"], f["R"]), f["gx"])
        assert chunks >= 3, ("not in steady state", line, chunks)


def assert_pf_steady(line, nr):
    name, f = line
    assert name == "eval_values_pf_kernel" and f["NR"] == nr, (line, nr)
    assert per_cta(f["ntiles"], f["grid"]) >= 4, ("not in steady state", line)


def gram_lines(lines):
    return [x for x in lines if x[0] in ("gram_mma_kernel", "gram_kernel")]


def pf_lines(lines):
    return [x for x in lines if x[0] == "eval_values_pf_kernel"]


# ------------------------------------------------------------------------------------------------
# A. exact Gram on integer data
# ------------------------------------------------------------------------------------------------
def M(st, multi, guard, gen):
    return ("mma", st, multi, guard, gen)


def R(t):
    return ("reg", t)


# Switches that leave the form alone but change the ring: depth 2 (the parity flips every second chunk), 32-row chunks.
RING = ({"VS_GRAM_STAGES": 2}, {"VS_GRAM_RC": 32})

# (id, k, l, row counts, offset of the values in a NaN-padded device buffer (elements), runs)
#   runs: (switches, form with the second-order block, form without it, row counts the run applies to); a form of "reg" only
#   checks that the register-tile kernel ran.  Row counts: an even one (l = 1: the plain form) and an odd one (GEN form; the
#   runs of odd value blocks start 8 bytes off a 16-byte boundary when rows * l is odd).
def _nonmulti(k, rows, st, guard2):
    runs = [({}, M(st, 0, guard2, 0), M(st, 0, 1, 0), (rows,)), ({}, M(st, 0, guard2, 1), M(st, 0, 1, 1), (rows + 1,))]
    runs += [(env, M(st, 0, guard2, g), M(st, 0, 1, g), (r,)) for env in RING for g, r in ((0, rows), (1, rows + 1))]
    runs += [({"VS_GRAM_MMA": 0}, "reg", "reg", (rows, rows + 1))]
    return ("k%d" % k, k, 1, (rows, rows + 1), 0, runs)


def _multi(k, l, rows, st2, st1, extra=()):
    gens = ((l > 1 and 1 or 0, rows), (1, rows + 1))
    runs = [({}, M(st2, 1, 1, g), M(st1, 1, 1, g), (r,)) for g, r in gens]
    runs += [(env, M(st2, 1, 1, g), M(st1, 1, 1, g), (r,)) for env in RING for g, r in gens]
    runs += [({"VS_GRAM_MMA": 0}, "reg", "reg", (rows, rows + 1))] + list(extra)
    return ("k%d-l%d" % (k, l), k, l, (rows, rows + 1), 0, runs)


GRAM_CASES = [
    _nonmulti(3, 1 << 21, 2, 1),                     # (up to two CTAs per SM: twice the rows)
    _nonmulti(4, 1 << 20, 2, 0),
    _nonmulti(10, 1 << 20, 3, 0),
    _nonmulti(14, 1 << 19, 4, 0),
    _nonmulti(17, 1 << 19, 6, 1),
    _nonmulti(20, 1 << 20, 6, 0),
    _multi(20, 3, 1 << 18, 4, 4, extra=[
        ({"VS_GRAM_ST": 2}, M(2, 1, 1, 1), M(2, 1, 1, 1), (1 << 18, (1 << 18) + 1)),                 # three passes
        ({"VS_GRAM_ST": 2, "VS_GRAM_WARPS": 31}, M(2, 1, 1, 1), M(2, 1, 1, 1), ((1 << 18) + 1,)),    # two passes
        ({"VS_GRAM_GEN": 0}, "reg", "reg", (1 << 18, (1 << 18) + 1))]),
    _multi(24, 1, 1 << 19, 4, 4),
    _multi(50, 1, 1 << 18, 2, 4, extra=[
        ({"VS_GRAM_WARPS": 15}, M(2, 1, 1, 0), M(4, 1, 1, 0), (1 << 18,)),                           # two passes
        ({"VS_GRAM_ST": 4}, M(4, 1, 1, 0), M(4, 1, 1, 0), (1 << 18,)),
        ({"VS_GRAM_ST": 4}, M(4, 1, 1, 1), M(4, 1, 1, 1), ((1 << 18) + 1,))]),
    _multi(100, 1, (1 << 17) + 2, 4, 4),
    _multi(1, 16, 3 << 16, 4, 4),                    # the largest l of the tensor path
    # l > 16: the shifted sums do not fit super-tile (0, 0) -> register-tile kernel, every tile size it can pick
    ("k1-l17", 1, 17, (65537,), 0, [({}, R(8), R(6), (65537,))]),
    ("k1-l64", 1, 64, (65537,), 0, [({}, R(4), R(6), (65537,))]),
    ("k2-l33", 2, 33, (65537,), 0, [({}, R(4), R(4), (65537,))]),
    # values 8 bytes off a 16-byte boundary: no bulk copies -> register-tile kernel without a switch
    ("k5-l3-misaligned", 5, 3, (180001,), 1, [({}, R(6), R(4), (180001,))]),
]


def _mma_instantiations():
    """The 20 gram_mma_kernel instantiations of launch_gram_mma (VS_MMA_CASE)."""
    out = {M(st, 0, guard, gen) for st in (2, 3, 4, 6) for guard in (0, 1) for gen in (0, 1)}
    return out | {M(st, 1, 1, gen) for st in (4, 2) for gen in (0, 1)}


def test_gram_cases_cover_every_form():
    """The cases below between them run all 20 tensor-path instantiations and each tile size T in {4, 6, 8} that
    make_geom / geom_cost can pick for l <= 64 (every one of them can be picked).  Each case checks from the trace that the
    form listed here is the one that ran."""
    seen = set()
    for case in GRAM_CASES:
        for env, f2, f1, rows in case[5]:
            seen |= {f for f in (f2, f1) if f != "reg"}
    want = _mma_instantiations() | {R(4), R(6), R(8)}
    assert len(_mma_instantiations()) == 20
    assert seen == want, (sorted(want - seen), sorted(seen - want))


def _integer_values(k, l, rows, seed):
    """Integer values in [-512, 511] as float64, Objective.flat() layout (row t * rows + r, column o)."""
    rng = numpy.random.RandomState(seed)
    return rng.randint(-512, 512, size=((2 + 2 * k) * rows, l)).astype(numpy.float64)


def exact_partials(k, l, rows, vals):
    """Partial sums of partials_from_values with shift = the first row, computed so that every sum is exact: integers of
    magnitude <= 512 give products <= 2^18 and shifted squares < 2^20, so with rows < 2^33 every partial sum of any
    summation order stays below 2^53 and is exact -- DMMA, DFMA and BLAS alike."""
    assert numpy.abs(vals).max() <= 512 and rows < 2 ** 33
    nt = 2 + 2 * k
    m = nt * l
    V = vals[:nt * rows].reshape(nt, rows, l).transpose(0, 2, 1).reshape(m, rows)     # coordinate-major
    shift = vals[0]
    d = V[:2 * l] - numpy.concatenate([shift, shift])[:, None]
    G = V @ V.T
    return numpy.concatenate([d.sum(axis=1), (d * d).sum(axis=1), G[numpy.triu_indices(m)]]), shift


@pytest.mark.parametrize("case", GRAM_CASES, ids=[c[0] for c in GRAM_CASES])
def test_gram_exact_in_steady_state(ctx, monkeypatch, tmp_path, case):
    """Every form equals the exact partial sums bit for bit, with and without the second-order block (first 2l Gram rows),
    reading its values from the middle of a NaN-padded device buffer and writing between NaN guards: a chunk counted twice
    or skipped, a stale stage, a read past a run or a write outside the output shows.  indices_from_values is bit-identical
    to the estimators of the exact partial sums (same shift)."""
    import torch
    name, k, l, row_counts, offset, runs = case
    trace = Tracer(ctx, monkeypatch, tmp_path)
    nt = 2 + 2 * k
    m = nt * l
    top = max(row_counts)
    host = _integer_values(k, l, top, seed=1000 * k + l)
    dev = torch.full((host.size + 2 * PAD,), float("nan"), dtype=torch.float64, device="cuda")
    dev[PAD + offset:PAD + offset + host.size] = torch.from_numpy(host.ravel()).cuda()
    plen = 4 * l + m * (m + 1) // 2
    first = 4 * l + sum(m - p for p in range(2 * l))                 # sums + Gram rows p < 2l: what first-order mode computes
    out = torch.full((plen + 2 * PAD,), float("nan"), dtype=torch.float64, device="cuda")
    for rows in row_counts:
        vals = host[:nt * rows]                      # the values of `rows` rows are a prefix of the buffer (row t * rows + r)
        ref, shift = exact_partials(k, l, rows, vals)
        fv = dev[PAD + offset:PAD + offset + nt * rows * l]
        for env, f2, f1, applies in runs:
            if rows not in applies:
                continue
            for flags, want_form in ((SO, f2), (0, f1)):
                out.fill_(float("nan"))
                _, lines = trace(lambda: ctx.partials_from_values(k, l, rows, fv, shift=shift, flags=flags,
                                                                  out=out[PAD:PAD + plen]), **env)
                what = (name, rows, env, flags)
                got = out.cpu().numpy()
                assert numpy.isnan(got[:PAD]).all() and numpy.isnan(got[PAD + plen:]).all(), what
                got = got[PAD:PAD + plen]
                lines = gram_lines(lines)
                assert len(lines) == 1, (what, lines)
                if want_form == "reg":
                    assert lines[0][0] == "gram_kernel", (what, lines)
                else:
                    assert form(lines[0]) == want_form, (what, lines)
                if lines[0][0] == "gram_mma_kernel":
                    f = lines[0][1]
                    assert f["oddrun"] == (rows * l) % 2 and f["second"] == flags, (what, lines)
                    if "VS_GRAM_STAGES" in env:
                        assert f["nstage"] == 2, (what, lines)
                    if "VS_GRAM_RC" in env:
                        assert f["rc"] == 32, (what, lines)
                assert_gram_steady(lines[0])
                n_cmp = plen if flags else first
                bad = numpy.flatnonzero(got[:n_cmp] != ref[:n_cmp])
                assert bad.size == 0, (what, lines, bad[:8], got[bad[:8]], ref[bad[:8]])
        # indices_from_values (shift = the first row as well) against the estimators of the exact partial sums
        res = ctx.indices_from_values(k, l, rows, rows, fv)
        want = ctx.finalize(k, l, rows, ref)
        for nm in NAMES:
            assert (getattr(res, nm) == getattr(want, nm)).all(), (name, rows, nm)


# ------------------------------------------------------------------------------------------------
# B. contract tolerance at the documented sizes
# ------------------------------------------------------------------------------------------------
def assert_indices(res, ref, names=NAMES, what=""):
    for nm in names:
        try:
            close(numpy.asarray(getattr(res, nm)).reshape(numpy.shape(ref[nm])), ref[nm])
        except AssertionError as e:
            raise AssertionError("%s %s: %s" % (what, nm, e))


def test_indices_from_values_documented_size(ctx, monkeypatch, tmp_path):
    """k = 20, n = 2^22 (the configuration DESIGN.md §4.3 times): the g-function's values through indices_from_values
    against the oracle and against the fused kernel on the same design, bit-reproducible run to run."""
    import torch
    trace = Tracer(ctx, monkeypatch, tmp_path)
    k, n = 20, 1 << 22
    a = gparams(k)
    vals = torch.from_numpy(cport.values(k, n, GF, a)).cuda()
    res, lines = trace(lambda: ctx.indices_from_values(k, 1, n, n, vals))
    lines = gram_lines(lines)
    assert len(lines) == 1 and form(lines[0]) == M(6, 0, 0, 0), lines
    assert_gram_steady(lines[0])
    again = ctx.indices_from_values(k, 1, n, n, vals)
    for nm in NAMES:
        assert (getattr(again, nm) == getattr(res, nm)).all(), nm
    del vals
    assert_indices(res, cport.run(k, n, GF, a), what="oracle")
    fused = ctx.run_fused(k, n, perm_of(n), GF, a)
    assert_indices(res, {nm: numpy.asarray(getattr(fused, nm)) for nm in NAMES}, what="fused")


def test_indices_from_values_trimmed_rows(ctx, monkeypatch, tmp_path):
    """rows = n - 3 (NaN rows trimmed: the divisors stay n and n - 1) in the odd-row form, against the estimators in extended
    precision."""
    trace = Tracer(ctx, monkeypatch, tmp_path)
    k, n = 20, 1 << 19
    rows = n - 3
    vals = cport.values(k, n, GF, gparams(k), i1=rows)
    res, lines = trace(lambda: ctx.indices_from_values(k, 1, n, rows, vals))
    lines = gram_lines(lines)
    assert len(lines) == 1 and form(lines[0]) == M(6, 0, 0, 1), lines
    assert_gram_steady(lines[0])
    ex = oexact.indices(vals.reshape(-1, 1), k, n, rows)
    assert_indices(res, ex, what="exact")


# ------------------------------------------------------------------------------------------------
# C. product-form values and the two-phase route
# ------------------------------------------------------------------------------------------------
def _sources(k, n):
    """(name, kwargs of ctx.eval_values, kwargs of cport.values): identity; linear scaling with a discard; raw points."""
    from varsens_b200 import _cabi
    lb, ub = numpy.linspace(0.05, 0.3, k), numpy.linspace(0.6, 0.97, k)
    raw = numpy.random.RandomState(k).rand(2 * n, k)
    return (("identity", {}, {}),
            ("linear", dict(discard=777, scale=_cabi.Scale(_cabi.SCALE_LINEAR, lb, ub)), dict(discard=777, scale=("linear", lb, ub))),
            ("raw", dict(raw=raw), dict(raw=raw)))


@pytest.mark.parametrize("k", (24, 50, 100))
def test_eval_values_product_form_steady_state(ctx, monkeypatch, tmp_path, k):
    """eval_values_pf_kernel with >= 4 tiles per CTA (the next tile's permutation entry is prefetched) and a ragged last
    tile: against the oracle at rtol 1e-13; 64-row tiles (VS_PF_ROWS=64, NR = 2) bit-identical to 32-row tiles, because each
    row's arithmetic is the same; a window bit-identical to the same slice of the whole run; the point-by-point kernel
    (VS_NO_PF_EVAL=1) within rtol 1e-13.  At k = 100 the 64-row tiles do not fit shared memory and the 32-row form runs."""
    trace = Tracer(ctx, monkeypatch, tmp_path)
    n = (1 << 16) + 5
    a, p = gparams(k), perm_of(n)
    nr2 = 2 if k <= 50 else 1
    lo, hi = 12345, n - 7
    for name, kw, okw in _sources(k, n):
        want = cport.values(k, n, GF, a, **okw)
        whole, lines = trace(lambda: ctx.eval_values(k, n, p, GF, a, **kw))
        assert len(pf_lines(lines)) == 1, (name, lines)
        assert_pf_steady(pf_lines(lines)[0], 1)
        numpy.testing.assert_allclose(whole, want, rtol=1e-13, atol=0, err_msg=name)
        wide, lines = trace(lambda: ctx.eval_values(k, n, p, GF, a, **kw), VS_PF_ROWS=64)
        assert_pf_steady(pf_lines(lines)[0], nr2)
        assert (wide == whole).all(), (name, int((wide != whole).sum()))
        for env, nr in (({}, 1), ({"VS_PF_ROWS": 64}, nr2)):
            win, lines = trace(lambda: ctx.eval_values(k, n, p, GF, a, i_begin=lo, i_end=hi, **kw), **env)
            assert_pf_steady(pf_lines(lines)[0], nr)
            assert (win == whole[:, lo:hi]).all(), (name, env, int((win != whole[:, lo:hi]).sum()))
        slow, lines = trace(lambda: ctx.eval_values(k, n, p, GF, a, **kw), VS_NO_PF_EVAL=1)
        assert not pf_lines(lines), (name, lines)
        numpy.testing.assert_allclose(slow, want, rtol=1e-13, atol=0, err_msg=name)
        numpy.testing.assert_allclose(whole, slow, rtol=1e-13, atol=0, err_msg=name)


@pytest.mark.parametrize("k", (24, 50))
def test_two_phase_route_steady_state(ctx, monkeypatch, tmp_path, k):
    """run_fused at k > 20 (values to HBM, then the Gram kernel) against the oracle; three ragged shards with a host
    permutation, two of them with i_begin != 0 (the shared shift f(M_1[0]) is evaluated separately for those), add up to
    the whole and finalize to the oracle's indices."""
    trace = Tracer(ctx, monkeypatch, tmp_path)
    n = 1 << 18
    a, p = gparams(k), perm_of(n)
    want = cport.run(k, n, GF, a)
    res, lines = trace(lambda: ctx.run_fused(k, n, p, GF, a))
    assert len(pf_lines(lines)) == 1 and len(gram_lines(lines)) == 1, lines
    assert_pf_steady(pf_lines(lines)[0], 1)
    assert_gram_steady(gram_lines(lines)[0])
    assert_indices(res, want, what="run_fused")
    whole = ctx.fused_partials(k, n, p, GF, a)
    acc = numpy.zeros_like(whole)
    for lo, hi in ((0, 100003), (100003, 100004), (100004, n)):
        acc += ctx.fused_partials(k, n, p, GF, a, i_begin=lo, i_end=hi)
    numpy.testing.assert_allclose(acc, whole, rtol=1e-12, atol=1e-9)
    assert_indices(ctx.finalize(k, 1, n, acc), want, what="shards")
