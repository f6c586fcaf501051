"""Timings and accuracy of the adaptive mass-action network objective (VS_OBJ_MASS_ACTION_ADAPTIVE,
csrc/kernels_network.cu: network_adaptive_kernel) beside the fixed-step one.  Prints one JSON document:
  mid_network   the seeded network of tools/bench_mass_action.py (seed 2024, S=32, R=48, L=4, k=64, n=2^14, linear scaling
                [0.5, 2]) over t in (0, 10] with 4 output times, at rtol 1e-6 and 1e-9: kernel ms, trajectories/s, the four
                step counts and the lane utilisation; the max abs error of the final-time observables against a
                tight-tolerance reference (the oracle's restatement at rtol 1e-12, atol 1e-15) on sampled design points.
                Beside it the fixed-step kernel at dt = 0.01, 1000 steps, and its error against the same reference.
  fast_pair     a slower seeded network plus one reversible pair with rates 1e3: the fixed step at dt = 0.01 is unstable
                (rate x dt beyond RK4's bound) and gives non-finite values, the adaptive one is finite and within tolerance.
  c5_chain      the C5 chain (k=20, n=2^18, magnitude scaling) as an adaptive network against RK4Chain<10> (dt = 0.01, 1000
                steps): both kernel times and their agreement; and the chain as a fixed-step network (the r03 record).
Needs a CUDA device (the library has no CPU fallback).  Run:  python tools/bench_mass_action_adaptive.py > adaptive.json"""
import json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy, torch
import varsens_b200 as vb
from varsens_b200 import _cabi
from oracle import mass_action as ob

if not torch.cuda.is_available():
    raise SystemExit("bench_mass_action_adaptive: no CUDA device")
ctx = vb.Context.get(0)
ctx.set_timing(True)
ctx.set_stream(torch.cuda.current_stream().cuda_stream)
dev = torch.device("cuda", 0)
out = {"gpu": torch.cuda.get_device_name(0)}
q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                   stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30)
out["power_limit_and_max_sm_clock"] = q.stdout.strip()
MAA, MA = _cabi.OBJ_MASS_ACTION_ADAPTIVE, _cabi.OBJ_MASS_ACTION


def perm_dev(n):
    return torch.from_numpy(numpy.random.RandomState(1).permutation(n).astype(numpy.int32)).to(dev)


def kernel_ms(fn, reps=2, warm=1):
    """Median device time of the evaluation kernel (CUDA events the library records around it)."""
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        fn()
        torch.cuda.synchronize()
        ts.append(ctx.last_kernel_ms())
    return float(numpy.median(ts))


def sampled(k, n, p, scale, count=256):
    """(flat row indices, scaled points) of `count` design rows from each of three blocks (M_1, N_j[0], N_nj[k-1])."""
    idx = numpy.concatenate([numpy.arange(b * n, b * n + count) for b in (0, 2, 1 + 2 * k)])
    pts = numpy.concatenate([ctx.sample_flat(k, n, p, scale=scale, row_begin=b * n, row_end=b * n + count)
                             for b in (0, 2, 1 + 2 * k)])
    return idx, pts


def adaptive_run(k, n, p, scale, par, idx, ref_final, L):
    traj = 2 * n * (1 + k)
    l = int(par[2]) * int(par[3])
    v = torch.empty(traj * l, dtype=torch.float64, device=dev)
    ms = kernel_ms(lambda: ctx.eval_values(k, n, p, MAA, par, scale=scale, out=v))
    st = ctx.network_stats()
    vals = v.view(traj, l)[torch.from_numpy(idx).to(dev)].cpu().numpy()
    return {"rtol": float(par[4]), "atol": float(par[5]), "kernel_ms": ms, "trajectories_per_s": traj / (ms * 1e-3),
            "stats": st, "lane_utilisation": (st["accepted"] + st["rejected"]) / st["lane_work"],
            "steps_per_trajectory": st["accepted"] / traj, "values_finite": bool(torch.isfinite(v).all()),
            "max_abs_err_final_time": float(numpy.abs(vals[:, -L:] - ref_final).max())}


def fixed_run(k, n, p, scale, par, idx, ref_final):
    traj = 2 * n * (1 + k)
    L = int(par[2])
    v = torch.empty(traj * L, dtype=torch.float64, device=dev)
    ms = kernel_ms(lambda: ctx.eval_values(k, n, p, MA, par, scale=scale, out=v))
    vals = v.view(traj, L)[torch.from_numpy(idx).to(dev)].cpu().numpy()
    fin = bool(torch.isfinite(v).all())
    return {"dt": float(par[3]), "nsteps": int(par[4]), "kernel_ms": ms, "trajectories_per_s": traj / (ms * 1e-3),
            "values_finite": fin, "max_abs_err_final_time": float(numpy.abs(vals - ref_final).max()) if fin else None}


# ---- 1. the r03 mid network over (0, 10]
k, n, S, R, L = 64, 1 << 14, 32, 48, 4
times = [2.5, 5.0, 7.5, 10.0]
mid = ob.random_network(2024, S, R, L, k, dt=0.01, nsteps=1000)
p = perm_dev(n)
scl = _cabi.Scale(_cabi.SCALE_LINEAR, numpy.full(k, 0.5), numpy.full(k, 2.0))
idx, pts = sampled(k, n, p, scl)
ref = ob.points_values(pts, ob.adaptive_of(mid, times, rtol=1e-12, atol=1e-15))[0][:, -L:]
out["mid_network"] = {"S": S, "R": R, "L": L, "k": k, "n": n, "times": times, "trajectories": 2 * n * (1 + k),
                      "reference": "oracle restatement at rtol 1e-12, atol 1e-15", "sampled_points": len(idx),
                      "adaptive": [adaptive_run(k, n, p, scl, ob.adaptive_of(mid, times, rtol=rt, atol=rt * 1e-3), idx, ref, L)
                                   for rt in (1e-6, 1e-9)],
                      "fixed_step": fixed_run(k, n, p, scl, mid, idx, ref)}

# ---- 2. a fast reversible pair the fixed step cannot integrate at dt = 0.01
k, n, S, R, L = 8, 1 << 12, 8, 12, 2
net = ob.unpack(ob.random_network(7, S, R, L, k, dt=0.01, nsteps=1000), adaptive=False)
pair = [0, -1, 1, -1, -1, 1000.0, -1, 800.0]                       # X_0 <-> X_1, kf + kr = 1800: 18 x dt, RK4's bound is 2.8
net.rec = numpy.vstack([net.rec, pair])
fast = ob.pack(net)
p = perm_dev(n)
scl = _cabi.Scale(_cabi.SCALE_LINEAR, numpy.full(k, 0.5), numpy.full(k, 2.0))
idx, pts = sampled(k, n, p, scl)
ref = ob.points_values(pts, ob.adaptive_of(fast, [10.0], rtol=1e-12, atol=1e-15))[0]
out["fast_pair"] = {"S": S, "R": R + 1, "L": L, "k": k, "n": n, "times": [10.0], "pair_rates": [1000.0, 800.0],
                    "reference_max_abs": float(numpy.abs(ref).max()),
                    "adaptive": adaptive_run(k, n, p, scl, ob.adaptive_of(fast, [10.0], rtol=1e-6, atol=1e-9), idx, ref, L),
                    "fixed_step": fixed_run(k, n, p, scl, fast, idx, ref)}

# ---- 3. the C5 chain as an adaptive network against RK4Chain<10>, and as a fixed-step network
k, n, steps = 20, 1 << 18, 1000
p = perm_dev(n)
r = numpy.array([1.0] * 10 + [0.5] * 10)
sc = _cabi.Scale(_cabi.SCALE_POWER, r / 10.0, r * 10.0)
traj = 2 * n * (1 + k)
va = torch.empty(traj, dtype=torch.float64, device=dev)
vn = torch.empty(traj, dtype=torch.float64, device=dev)
ms_chain = kernel_ms(lambda: ctx.eval_values(k, n, p, _cabi.OBJ_RK4_CHAIN, [0.01, steps], scale=sc, out=va))
ms_fixed = kernel_ms(lambda: ctx.eval_values(k, n, p, MA, ob.chain_network(10, 0.01, steps), scale=sc, out=vn))
same = bool(torch.equal(va.view(torch.int64), vn.view(torch.int64)))
c5 = {"k": k, "n": n, "trajectories": traj, "rk4_chain_kernel_ms": ms_chain, "fixed_network_kernel_ms": ms_fixed,
      "fixed_network_bit_identical_to_chain": same, "adaptive": []}
for rt in (1e-6, 1e-9):
    par = ob.adaptive_of(ob.chain_network(10), [10.0], rtol=rt, atol=rt * 1e-3)
    ms = kernel_ms(lambda: ctx.eval_values(k, n, p, MAA, par, scale=sc, out=vn))
    st = ctx.network_stats()
    c5["adaptive"].append({"rtol": rt, "atol": rt * 1e-3, "kernel_ms": ms, "ratio_over_rk4_chain": ms / ms_chain, "stats": st,
                           "lane_utilisation": (st["accepted"] + st["rejected"]) / st["lane_work"],
                           "max_abs_diff_vs_rk4_chain": float((vn - va).abs().max())})
out["c5_chain"] = c5
print(json.dumps(out, indent=1))
