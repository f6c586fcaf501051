"""CPU-only checks of the boundary: the C-ABI library loads, exports every symbol the header declares,
its host-side tables equal the oracle's, and the host mirror's pure-Python logic (scale tracing,
sharding, the N>1 all-reduce plumbing over gloo) works.  No GPU compute is called here."""
import os
import re
import subprocess
import sys

import numpy
import pytest

from oracle import halton as ohalton, pipeline, cport, objectives as ob

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def cabi():
    import __graft_entry__ as g
    g.build()
    from varsens_b200 import _cabi
    return _cabi


def test_library_exports_every_declared_symbol(cabi):
    header = open(os.path.join(ROOT, "include", "varsens_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(vs_[a-z0-9_]+)\s*\(", header)))
    assert declared == sorted(cabi.SYMBOLS)
    lib = cabi.lib()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.vs_abi_version() == 1


def test_halton_term_table_equals_oracle(cabi):
    for k, mx in ((1, 10), (6, 121 + 2048), (20, 401 + 2 ** 25), (50, 1001 + 2 ** 23)):
        b, nd, off, t = cabi.halton_terms(k, mx)
        ob_, ond, ooff, ot = ohalton.halton_term_table(k, mx)
        assert (b == ob_).all() and (nd == ond).all() and (off == ooff).all()
        assert t.shape == ot.shape and (t == ot).all()
    assert cabi.halton_terms(20, 401 + 2 ** 25)[3].size == 3523          # SURVEY §7 probe


def test_partials_len(cabi):
    from varsens_b200 import dist
    for k, l in ((1, 1), (6, 1), (20, 1), (6, 2), (50, 3)):
        m = (2 + 2 * k) * l
        assert cabi.lib().vs_partials_len(k, l) == 4 * l + m * (m + 1) // 2 == dist.partials_layout(k, l)["length"]


def test_no_cpu_fallback(cabi):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(cabi.VarsensError, match="no CPU fallback"):
        cabi.Context(0)
    import varsens_b200 as vb
    with pytest.raises(cabi.VarsensError):
        vb.Varsens(vb.GFunction([0.0, 1.0]), lambda x: x, 2, 8, verbose=False)
    with pytest.raises(cabi.VarsensError, match="device functor"):
        vb.GFunction([0.0])(numpy.zeros(1))


def test_scale_helpers_match_reference_numbers(refgold):
    from varsens_b200 import scale
    p = refgold["scale_p"]
    assert (scale.linear(p, -3.5, 12.25) == refgold["scale_linear"]).all()
    assert (scale.power(p, 0.01, 250.0) == refgold["scale_power"]).all()
    assert (scale.percentage(p, 40.0, 33.0) == refgold["scale_percentage"]).all()
    assert (scale.magnitude(p, 2.5, 2.0, 10.0) == refgold["scale_magnitude"]).all()
    import varsens_b200 as vb
    assert vb.linear is scale.linear and vb.magnitude is scale.magnitude          # star export, __init__.py:2


def test_scale_tracing(cabi):
    from varsens_b200 import scale
    lb, ub = numpy.array([-1.0, 2.0, 3.0]), numpy.array([1.0, 4.0, 30.0])
    d = scale.trace(lambda x: x, 3)
    assert d.kind == cabi.SCALE_IDENTITY
    d = scale.trace(lambda x: scale.linear(x, lb, ub), 3)
    assert d.kind == cabi.SCALE_LINEAR and (d.lower == lb).all() and (d.upper == ub).all()
    d = scale.trace(lambda x: scale.percentage(x, ub, 33.0), 3)
    assert d.kind == cabi.SCALE_LINEAR and numpy.allclose(d.lower, ub * 0.67)
    d = scale.trace(lambda x: scale.magnitude(x, ub, orders=1.0), 3)
    assert d.kind == cabi.SCALE_POWER and (d.lower == ub / 10.0).all() and (d.upper == ub * 10.0).all()
    d = scale.trace(lambda x: scale.linear(x, -numpy.pi, numpy.pi), 3)            # scalar bounds broadcast
    assert d.kind == cabi.SCALE_LINEAR and d.lower.shape == (3,)
    assert scale.trace(lambda x: scale.linear(x, lb, ub) + 1.0, 3) is None       # not a pure scale.* call
    assert scale.trace(lambda x: x * 2.0, 3) is None
    assert scale.trace(lambda x: numpy.sqrt(x), 3) is None


def test_negative_discard_is_rejected():
    """The C ABI takes discard unsigned and ctypes wraps -1 around to 2^64 - 1, which would move the first Halton index to 0;
    the binding refuses it instead (a traced scaling creates no context, so this needs no GPU)."""
    import varsens_b200 as vb
    with pytest.raises(vb.VarsensError, match="discard"):
        vb.Sample(6, 8, lambda x: x, discard=-1)
    from varsens_b200 import _cabi
    assert _cabi.discard_arg(0) == 0 and _cabi.discard_arg(7) == 7


def test_shard_range_partitions():
    from varsens_b200 import dist
    for total in (0, 1, 7, 1024, 2 ** 24 + 5):
        for ws in (1, 2, 3, 8):
            edges = [dist.shard_range(total, r, ws) for r in range(ws)]
            assert edges[0][0] == 0 and edges[-1][1] == total
            assert all(edges[i][1] == edges[i + 1][0] for i in range(ws - 1))
            sizes = [hi - lo for lo, hi in edges]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        dist.shard_range(10, 2, 2)


_WORKER = r"""
import os, sys, numpy, torch, torch.distributed as dist
sys.path.insert(0, {root!r})
from varsens_b200 import dist as vdist
from oracle import cport, pipeline
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
k, n = 6, 1000
a = [0, .5, 3, 9, 99, 99]
rank, ws = vdist.world()
lo, hi = vdist.shard_range(n, rank, ws)
S = cport.sums(k, n, cport.OBJ_GFUNCTION, a, i0=lo, i1=hi)           # this rank's shard, oracle arithmetic
lay = vdist.partials_layout(k)
p = numpy.zeros(lay["length"])
m, J, N = lay["m"], range(2, 2 + k), range(2 + k, 2 + 2 * k)
g = lay["gram"]
p[lay["S_A"]], p[lay["S_B"]], p[lay["Q_A"]], p[lay["Q_B"]] = S["s_a"], S["s_b"], S["q_a"], S["q_b"]
p[g(0, 1)] = S["s_ab"]; p[g(0, 0)] = S["q_a"]; p[g(1, 1)] = S["q_b"]
for j in range(k):
    p[g(0, 2 + j)], p[g(1, 2 + k + j)], p[g(0, 2 + k + j)], p[g(1, 2 + j)] = S["aJ"][j], S["bN"][j], S["aN"][j], S["bJ"][j]
    for i in range(k):
        p[g(2 + k + i, 2 + j)] = S["NJ"][i, j]
        if i <= j:
            p[g(2 + k + i, 2 + k + j)] = S["NN"][i, j]; p[g(2 + i, 2 + j)] = S["JJ"][i, j]
t = torch.from_numpy(p)
vdist.allreduce_partials(t)
if rank == 0:
    whole = cport.sums(k, n, cport.OBJ_GFUNCTION, a)
    q = t.numpy()
    assert abs(q[g(0, 1)] - float(whole["s_ab"])) < 1e-9
    assert abs(q[g(2 + k + 1, 2 + 3)] - float(whole["NJ"][1, 3])) < 1e-9
    assert abs(q[lay["S_A"]] + q[lay["S_B"]] - float(whole["s_a"] + whole["s_b"])) < 1e-9
    print("GLOO_OK")
dist.destroy_process_group()
"""


def test_two_rank_allreduce_over_gloo(tmp_path):
    """world_size-2 run of the N>1 host path on CPU: shard ranges, partial-vector layout, one all-reduce."""
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT, port=port))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    outs = [p.communicate(timeout=180)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert "GLOO_OK" in outs[0]


def test_fast_digit_step_is_exact():
    """The multiply-only quotient/remainder step of the fused kernels (csrc/fused_impl.cuh digit_step) -- brute force."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "check_fastdiv.py")], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    assert r.returncode == 0, r.stdout.decode()[-2000:]


def test_sobol_direction_numbers_match_oracle():
    from varsens_b200 import sobol as vsobol
    from oracle import sobol as osobol
    assert (vsobol.joe_kuo_direction_numbers(40) == osobol.joe_kuo_direction_numbers(40)).all()


def test_objective_binary_batches_round_trip(tmp_path):
    """Objective.export/load with postfix='.npy' (SURVEY.md §8f.2): host-only path, exact round trip, and the
    reference's text format still reads back to 17 significant digits."""
    import math
    import varsens_b200 as vb
    k, n = 3, 40
    rng = numpy.random.RandomState(5)
    vals = rng.rand(2 * n * (1 + k), 2)
    o = vb.Objective(k, n, objective_vals=vals, verbose=False)
    o.export(str(tmp_path), "obj", ".npy", 100)
    nfiles = int(math.ceil(len(vals) / 100.0))
    assert sorted(p.name for p in tmp_path.iterdir()) == sorted("obj_%d.npy" % (i + 1) for i in range(nfiles))
    o2 = vb.Objective(k, n, verbose=False, indir=str(tmp_path), prefix="obj", postfix=".npy", nFiles=nfiles)
    assert (o2.flat() == vals).all()
    assert (o2.fN_nj == o.fN_nj).all() and o2.fN_j.shape == (k, n, 2)
    o.export(str(tmp_path), "objt", ".txt", 100)
    o3 = vb.Objective(k, n, verbose=False, indir=str(tmp_path), prefix="objt", postfix=".txt", nFiles=nfiles)
    assert (o3.flat() == vals).all()           # %.18e round-trips a double exactly
    with pytest.raises(Exception, match="Cannot find input file"):
        vb.Objective(k, n, verbose=False, indir=str(tmp_path), prefix="nope", postfix=".npy", nFiles=1)


def test_reference_permutation_cache_keeps_rng_side_effect():
    """saltelli.py:100-101 reseeds and advances numpy's GLOBAL legacy RNG; the cached permutation must leave it in the
    same state as a fresh draw, and equal the oracle's permutation."""
    from varsens_b200 import saltelli as vsalt
    vsalt._perm_cache.clear()
    for n in (1000, 1, 2, 4097):
        numpy.random.seed(12345)
        first = vsalt._reference_permutation(n)
        after_first = numpy.random.random_sample(3)
        numpy.random.seed(999)
        again = vsalt._reference_permutation(n)                 # cache hit
        after_again = numpy.random.random_sample(3)
        idx = numpy.arange(n)
        numpy.random.seed(1)
        numpy.random.shuffle(idx)
        want_after = numpy.random.random_sample(3)
        assert (first == idx).all() and again is first and first.dtype == numpy.uint32
        assert (first == pipeline.permutation(n)).all()
        assert (after_first == want_after).all() and (after_again == want_after).all()
    for n in range(10, 20):                                      # bounded: only the newest few are kept
        vsalt._reference_permutation(n)
    assert len(vsalt._perm_cache) <= 4


def test_c_permutation_equals_numpy_legacy_shuffle(cabi):
    """vs_reference_permutation (MT19937 + masked-rejection rk_interval on uint32, look-ahead prefetch) against the
    reference's own call, numpy.random.seed(1); numpy.random.shuffle (saltelli.py:100-101): the permutation, shuffling a
    2-D matrix (what the reference shuffles), and the generator state it leaves behind."""
    for n in list(range(0, 70)) + [127, 128, 129, 255, 256, 257, 1000, 4095, 4096, 4097, 65535, 65536, 65537, 1 << 20, (1 << 20) + 3]:
        perm, state = cabi.reference_permutation(n, 1)
        idx = numpy.arange(n)
        numpy.random.seed(1)
        numpy.random.shuffle(idx)
        want_state = numpy.random.get_state()
        assert perm.dtype == numpy.uint32 and (perm == idx).all(), n
        assert state[2] == want_state[2] and (state[1] == want_state[1]).all(), n      # same position, same key
    for seed in (0, 7, 2 ** 32 - 1):
        perm, state = cabi.reference_permutation(5000, seed)
        m = numpy.arange(5000 * 3).reshape(5000, 3)
        numpy.random.seed(seed)
        numpy.random.shuffle(m)                                                        # 2-D: rows are shuffled, same draws
        assert (m[:, 0] // 3 == perm).all()
        numpy.random.set_state(state)
        a = numpy.random.random_sample(4)
        b = numpy.random.random_sample(4)
        numpy.random.seed(seed)
        numpy.random.shuffle(numpy.arange(5000))
        assert (numpy.random.random_sample(4) == a).all() and (numpy.random.random_sample(4) == b).all()


@pytest.mark.slow_cpu
def test_c_permutation_full_size(cabi):
    """n = 2^24 (BASELINE config 3): equal to numpy's legacy shuffle, first values as frozen in SURVEY.md App. D."""
    perm, state = cabi.reference_permutation(1 << 24, 1)
    assert perm[:5].tolist() == [1374744, 606845, 6252930, 11816538, 1572451]
    assert (perm == numpy.random.RandomState(1).permutation(1 << 24)).all()


def test_computed_halton_terms_equal_the_table(cabi):
    """fused_impl.cuh digit_step_arith: the double-double-reciprocal form of digit / b^(j+1) must reproduce the term table bit
    for bit -- every digit of every position a 32-bit index reaches -- in each term-table mode (host self check of the
    library, exhaustive) and here once more in Python for the default mode with exact rational arithmetic as the referee."""
    from fractions import Fraction
    lib = cabi.lib()
    for mode in (cabi.HALTON_DIVIDE, cabi.HALTON_RECIPROCAL, cabi.HALTON_RUNNING_RECIPROCAL):
        assert lib.vs_halton_arith_check(64, mode) == 1
    assert lib.vs_halton_arith_check(20, 99) == -1
    # independent referee: the table's DIVIDE terms are the correctly rounded quotients digit / b^(j+1)
    bases, nd, off, terms = cabi.halton_terms(20, 2 ** 32 - 1)
    checked = 0
    for d in (1, 5, 11, 19):
        b = int(bases[d])
        for j in range(int(nd[d])):
            for digit in range(b):
                t = float(terms[off[d] + j * b + digit])
                assert t == digit / float(b ** (j + 1))
                exact = Fraction(digit, b ** (j + 1))
                ulp = numpy.spacing(t) if t else 0.0
                assert abs(Fraction(t) - exact) <= Fraction(ulp) / 2               # correctly rounded
                checked += 1
    assert checked > 500


def test_halton_term_table_modes(cabi):
    """The three term-table arithmetics (enum vs_halton_mode) against the oracle's restatement of each."""
    from oracle import halton as oh
    for mode, name in ((cabi.HALTON_DIVIDE, "divide"), (cabi.HALTON_RECIPROCAL, "reciprocal"),
                       (cabi.HALTON_RUNNING_RECIPROCAL, "running_reciprocal")):
        bases, nd, off, terms = cabi.halton_terms(12, 10 ** 7, mode)
        want = oh.term_table(12, 10 ** 7, mode=name)
        assert (terms == want["terms"]).all() and (off == want["offsets"]).all() and (nd == want["ndigits"]).all()
    d, r = cabi.halton_terms(12, 10 ** 7, cabi.HALTON_DIVIDE)[3], cabi.halton_terms(12, 10 ** 7, cabi.HALTON_RECIPROCAL)[3]
    assert (d != r).any() and numpy.abs(d - r).max() < 2.3e-16                     # the modes really differ, by an ulp
    with pytest.raises(cabi.VarsensError):
        cabi.halton_terms(12, 100, cabi.HALTON_HORNER)


def test_quantlib_initializer_reader(tmp_path):
    """varsens_b200.sobol.quantlib_direction_numbers: parse QuantLib-style initialiser arrays (C source with a pointer table,
    C source without one, plain text) and run QuantLib's recurrence.  Pinned by writing scipy's Joe-Kuo initialisers in those
    formats: the direction integers must equal the Joe-Kuo table the Sobol kernel is already pinned on."""
    import scipy
    from varsens_b200 import sobol as vsobol, _cabi
    z = numpy.load(os.path.join(os.path.dirname(scipy.__file__), "stats", "_sobol_direction_numbers.npz"))
    k = 40
    want = vsobol.joe_kuo_direction_numbers(k)
    inits = []
    for d in range(1, k):
        s_ = int(z["poly"][d]).bit_length() - 1
        inits.append([int(v) for v in z["vinit"][d][:s_]])
    names = ["dim%02dLevitanLemieuxinitializers" % (d + 2) for d in range(len(inits))]
    src = "// excerpt in the layout of ql/math/randomnumbers/sobolrsg.cpp\nnamespace {\n"
    for nm, m in zip(names, inits):
        src += "    static const unsigned long %s[] = {\n        %s, 0UL };\n" % (nm, ", ".join("%dUL" % v for v in m))
    decoy = "    static const unsigned long dim02Kuoinitializers[] = { 1UL, 0UL };\n"
    table = "    static const unsigned long * const LevitanLemieuxinitializers[%d] = {\n        %s\n    };\n}\n" % (
        len(names), ",\n        ".join(names))
    path = tmp_path / "sobolrsg.cpp"
    path.write_text(src + decoy + table)
    assert (vsobol.quantlib_direction_numbers(k, str(path)) == want).all()
    assert (vsobol.quantlib_direction_numbers(k, src + decoy, kind="LevitanLemieux") == want).all()       # no pointer table
    txt = "# dimension 2 onwards\n" + "\n".join(" ".join(str(v) for v in m) for m in inits)
    assert (vsobol.quantlib_direction_numbers(k, txt) == want).all()
    assert (vsobol.quantlib_direction_numbers(2, "1\n") == want[:2]).all()
    with pytest.raises(_cabi.VarsensError):
        vsobol.quantlib_direction_numbers(k, "1\n1 3\n")                                                 # too few dimensions
    with pytest.raises(_cabi.VarsensError):
        vsobol.quantlib_direction_numbers(3, "1\n2 3\n")                                                 # even initialiser


def test_header_enums_match_python_binding():
    """The ctypes binding hard-codes the header's enum values: parse include/varsens_b200.h and compare."""
    from varsens_b200 import _cabi
    text = open(os.path.join(ROOT, "include", "varsens_b200.h")).read()
    vals = {}
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    for body in re.findall(r"enum\s*\w*\s*\{([^}]*)\}", text):
        nxt = 0
        for item in body.split(","):
            item = item.strip()
            if not item:
                continue
            if "=" in item:
                name, v = [t.strip() for t in item.split("=")]
                nxt = int(v, 0)
            else:
                name = item
            vals[name] = nxt
            nxt += 1
    want = {"VS_MEM_HOST": _cabi.MEM_HOST, "VS_MEM_DEVICE": _cabi.MEM_DEVICE, "VS_SCALE_IDENTITY": _cabi.SCALE_IDENTITY,
            "VS_SCALE_LINEAR": _cabi.SCALE_LINEAR, "VS_SCALE_POWER": _cabi.SCALE_POWER, "VS_OBJ_GFUNCTION": _cabi.OBJ_GFUNCTION,
            "VS_OBJ_ISHIGAMI": _cabi.OBJ_ISHIGAMI, "VS_OBJ_RK4_CHAIN": _cabi.OBJ_RK4_CHAIN,
            "VS_FLAG_SECOND_ORDER": _cabi.FLAG_SECOND_ORDER, "VS_FLAG_SEPARABLE": _cabi.FLAG_SEPARABLE, "VS_OK": 0}
    for name, v in want.items():
        assert vals.get(name) == v, (name, vals.get(name), v)
    assert cport.OBJ_GFUNCTION == _cabi.OBJ_GFUNCTION and cport.OBJ_RK4_CHAIN == _cabi.OBJ_RK4_CHAIN     # oracle ids follow the ABI


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm) prints ONE JSON line with the contract's
    keys, times the oracle port on the host cores and needs no GPU; a non-zero rank under torchrun prints nothing and exits 0."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ)
    for key in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(key, None)
    p = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       cwd=root, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "evals/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["dtype"] == "f64" and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]
    env.update(RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    q = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       cwd=root, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert q.returncode == 0 and q.stdout.strip() == "", (q.stdout, q.stderr[-500:])


def test_bench_rejects_arguments_it_cannot_honour():
    """`--steps` is the number of timed steps, so it must be at least 1; `--dump-outputs` writes what the GPU arm computed and
    has nothing to write for the reference arm.  Both are refused before any work starts."""
    for extra in (["--steps", "0"], ["--impl", "reference", "--steps", "1", "--dump-outputs", "unused"]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, cwd=ROOT, stdout=subprocess.PIPE,
                           stderr=subprocess.PIPE, text=True, timeout=120)
        assert p.returncode == 2 and p.stdout == "" and "error:" in p.stderr, (extra, p.stderr[-500:])
