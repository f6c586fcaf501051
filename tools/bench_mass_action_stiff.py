"""Timings and accuracy of the stiff mass-action network objective (VS_OBJ_MASS_ACTION_STIFF, csrc/kernels_network.cu:
network_rosenbrock_kernel, Rodas3) beside the Dormand-Prince 5(4) one (VS_OBJ_MASS_ACTION_ADAPTIVE) on the same packed
descriptions, in the same call.  Prints one JSON document:
  fast_pair     tools/bench_mass_action_adaptive.py's network (seed 7, S=8, R=12, L=2, k=8, n=2^12, linear scaling [0.5, 2])
                plus one reversible pair X_0 <-> X_1, at rates 1e3 / 8e2 and 1e5 / 8e4, to t = 10 at rtol 1e-6, atol 1e-9
                (the explicit method's step is bound by stability, so its steps grow with the fastest rate; at 1e5 its
                trajectories are expected to exhaust max_steps = 100000 and fail).
  mid_network   the seeded network of tools/bench_mass_action.py (seed 2024, S=32, R=48, L=4, k=64, n=2^14) over (0, 10] with
                4 output times at rtol 1e-6, atol 1e-9: a non-stiff network, where the explicit method may well be faster.
For each method: kernel ms (CUDA events the library records around the kernel, median of 2 after 1 warm-up), trajectories/s,
the four step counts of vs_last_network_stats, the lane utilisation, and the max abs error of the final-time observables on
sampled design points against a tight reference: the oracle's Rodas3 at rtol 1e-12, atol 1e-15 for the fast pair (itself
checked against scipy's Radau at rtol 1e-12 on a few points), the oracle's Dormand-Prince at rtol 1e-12, atol 1e-15 for the
mid network.  Needs a CUDA device.  Run:  python tools/bench_mass_action_stiff.py > stiff.json"""
import json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy, torch
import varsens_b200 as vb
from varsens_b200 import _cabi
from oracle import mass_action as ob, mass_action_stiff as ost

if not torch.cuda.is_available():
    raise SystemExit("bench_mass_action_stiff: no CUDA device")
ctx = vb.Context.get(0)
ctx.set_timing(True)
ctx.set_stream(torch.cuda.current_stream().cuda_stream)
dev = torch.device("cuda", 0)
out = {"gpu": torch.cuda.get_device_name(0)}
q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                   stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30)
out["power_limit_and_max_sm_clock"] = q.stdout.strip()
METHODS = (("dopri5", _cabi.OBJ_MASS_ACTION_ADAPTIVE), ("rodas3", _cabi.OBJ_MASS_ACTION_STIFF))


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


def sampled(k, n, p, scale, count):
    """(flat row indices, scaled points) of `count` design rows from each of three blocks (M_1, N_j[0], N_nj[k-1])."""
    idx = numpy.concatenate([numpy.arange(b * n, b * n + count) for b in (0, 2, 1 + 2 * k)])
    pts = numpy.concatenate([ctx.sample_flat(k, n, p, scale=scale, row_begin=b * n, row_end=b * n + count)
                             for b in (0, 2, 1 + 2 * k)])
    return idx, pts


def run(objective, k, n, p, scale, par, idx, ref_final, L):
    traj = 2 * n * (1 + k)
    l = int(par[2]) * int(par[3])
    v = torch.empty(traj * l, dtype=torch.float64, device=dev)
    ms = kernel_ms(lambda: ctx.eval_values(k, n, p, objective, par, scale=scale, out=v))
    st = ctx.network_stats()
    vals = v.view(traj, l)[torch.from_numpy(idx).to(dev)].cpu().numpy()
    fin = numpy.isfinite(vals[:, -L:]).all(axis=1)
    return {"kernel_ms": ms, "trajectories_per_s": traj / (ms * 1e-3), "stats": st,
            "lane_utilisation": (st["accepted"] + st["rejected"]) / st["lane_work"],
            "accepted_per_trajectory": st["accepted"] / traj, "attempts_per_trajectory": (st["accepted"] + st["rejected"]) / traj,
            "values_finite": bool(torch.isfinite(v).all()),
            "max_abs_err_final_time": float(numpy.abs(vals[fin, -L:] - ref_final[fin]).max()) if fin.any() else None}


def both(k, n, p, scale, par, idx, ref_final, L):
    return {name: run(obj, k, n, p, scale, par, idx, ref_final, L) for name, obj in METHODS}


def radau_final(par, x):
    from scipy.integrate import solve_ivp
    net = ob.unpack(par, True)
    f, y0 = ob.numpy_rhs(par, x)
    sol = solve_ivp(f, (0.0, net.times[-1]), y0, method="Radau", t_eval=net.times[-1:], rtol=1e-12, atol=1e-14)
    return net.w @ sol.y[:, -1]


# ---- 1. the fast reversible pair at two rates
k, n, S, R, L = 8, 1 << 12, 8, 12, 2
p = perm_dev(n)
scl = _cabi.Scale(_cabi.SCALE_LINEAR, numpy.full(k, 0.5), numpy.full(k, 2.0))
idx, pts = sampled(k, n, p, scl, 64)
out["fast_pair"] = []
for kf, kr in ((1e3, 8e2), (1e5, 8e4)):
    net = ob.unpack(ob.random_network(7, S, R, L, k, dt=0.01, nsteps=1000), adaptive=False)
    net.rec = numpy.vstack([net.rec, [0, -1, 1, -1, -1, kf, -1, kr]])
    fast = ob.pack(net)
    ref = ost.points_values(pts, ob.adaptive_of(fast, [10.0], rtol=1e-12, atol=1e-15))[0]
    radau = numpy.array([radau_final(ob.adaptive_of(fast, [10.0]), x) for x in pts[:4]])
    par = ob.adaptive_of(fast, [10.0], rtol=1e-6, atol=1e-9)
    out["fast_pair"].append({"S": S, "R": R + 1, "L": L, "k": k, "n": n, "times": [10.0], "pair_rates": [kf, kr],
                             "rtol": 1e-6, "atol": 1e-9, "trajectories": 2 * n * (1 + k), "sampled_points": len(idx),
                             "reference": "oracle Rodas3 at rtol 1e-12, atol 1e-15",
                             "reference_vs_radau_max_abs": float(numpy.abs(ref[:4] - radau).max()),
                             **both(k, n, p, scl, par, idx, ref, L)})

# ---- 2. the mid network, not stiff
k, n, S, R, L = 64, 1 << 14, 32, 48, 4
times = [2.5, 5.0, 7.5, 10.0]
mid = ob.random_network(2024, S, R, L, k, dt=0.01, nsteps=1000)
p = perm_dev(n)
scl = _cabi.Scale(_cabi.SCALE_LINEAR, numpy.full(k, 0.5), numpy.full(k, 2.0))
idx, pts = sampled(k, n, p, scl, 256)
ref = ob.points_values(pts, ob.adaptive_of(mid, times, rtol=1e-12, atol=1e-15))[0][:, -L:]
par = ob.adaptive_of(mid, times, rtol=1e-6, atol=1e-9)
out["mid_network"] = {"S": S, "R": R, "L": L, "k": k, "n": n, "times": times, "rtol": 1e-6, "atol": 1e-9,
                      "trajectories": 2 * n * (1 + k), "nnz_lu": ost.stiff_sizes(par)["nlu"], "sampled_points": len(idx),
                      "reference": "oracle Dormand-Prince at rtol 1e-12, atol 1e-15", **both(k, n, p, scl, par, idx, ref, L)}
print(json.dumps(out, indent=1))
