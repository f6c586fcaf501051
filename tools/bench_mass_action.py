"""Timings of the mass-action network objective (VS_OBJ_MASS_ACTION, csrc/kernels_network.cu).  Prints one JSON document:
  c5_as_network   the C5 chain (k=20, n=2^18, dt=0.01, 1000 steps, magnitude scaling as in tools/bench_configs.py) written as
                  a network against OBJ_RK4_CHAIN: both evaluation-kernel times, their ratio, trajectories/s, bit-identity;
  mid_network     a seeded network, S=32, R=48 (orders 0-2), L=4, k=64, n=2^14, 1000 steps: kernel trajectories/s and the
                  end-to-end Varsens(...) time;
  torch_route     the same network as a @vectorized torch objective (RK4 written in torch) at a reduced n, for context.
Run on a B200:  python tools/bench_mass_action.py > mass_action.json"""
import json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy, torch
import varsens_b200 as vb
from varsens_b200 import _cabi, functors
from oracle import mass_action as ob

ctx = vb.Context.get(0)
ctx.set_timing(True)
ctx.set_stream(torch.cuda.current_stream().cuda_stream)
dev = torch.device("cuda", 0)
out = {"gpu": torch.cuda.get_device_name(0)}
try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30)
    out["power_limit_and_max_sm_clock"] = q.stdout.strip()
except Exception as exc:
    out["power_limit_and_max_sm_clock"] = "unavailable (%s)" % exc


def perm_dev(n):
    return torch.from_numpy(numpy.random.RandomState(1).permutation(n).astype(numpy.int32)).to(dev)


def kernel_ms(fn, reps=3, warm=1):
    """Median device time of the evaluation kernel (CUDA events the library records around it)."""
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        fn()
        torch.cuda.synchronize()
        ts.append(ctx.last_kernel_ms())
    return float(numpy.median(ts))


class Packed(functors.Functor):
    """A packed network description as a device functor (what MassActionNetwork.params returns)."""
    objective_id = _cabi.OBJ_MASS_ACTION

    def __init__(self, packed):
        self.packed = packed

    def params(self, k):
        return self.packed

    def outputs(self, k):
        return _cabi.objective_outputs(k, self.objective_id, self.packed)


# ---- 1. C5 written as a network against the register-resident RK4Chain<10>
k, n, steps = 20, 1 << 18, 1000
p = perm_dev(n)
ref = numpy.array([1.0] * 10 + [0.5] * 10)
sc = _cabi.Scale(_cabi.SCALE_POWER, ref / 10.0, ref * 10.0)
traj = 2 * n * (1 + k)
va = torch.empty(traj, dtype=torch.float64, device=dev)
vn = torch.empty(traj, dtype=torch.float64, device=dev)
chain = ob.chain_network(10, 0.01, steps)
ms_chain = kernel_ms(lambda: ctx.eval_values(k, n, p, _cabi.OBJ_RK4_CHAIN, [0.01, steps], scale=sc, out=va))
ms_net = kernel_ms(lambda: ctx.eval_values(k, n, p, _cabi.OBJ_MASS_ACTION, chain, scale=sc, out=vn))
torch.cuda.synchronize()
sl = slice(0, traj, 997)                                         # a sampled slice, compared bit for bit
same = bool(torch.equal(va[sl].view(torch.int64), vn[sl].view(torch.int64)))
out["c5_as_network"] = {"k": k, "n": n, "steps": steps, "trajectories": traj,
                        "rk4_chain_kernel_ms": ms_chain, "network_kernel_ms": ms_net, "ratio_network_over_chain": ms_net / ms_chain,
                        "rk4_chain_trajectories_per_s": traj / (ms_chain * 1e-3), "network_trajectories_per_s": traj / (ms_net * 1e-3),
                        "sampled_values": len(range(0, traj, 997)), "bit_identical_on_sample": same,
                        "all_values_bit_identical": bool(torch.equal(va.view(torch.int64), vn.view(torch.int64)))}
del va, vn

# ---- 2. seeded mid-size network
k, n, S, R, L = 64, 1 << 14, 32, 48, 4
mid = ob.random_network(2024, S, R, L, k, dt=0.01, nsteps=steps)
p = perm_dev(n)
lo, hi = numpy.full(k, 0.5), numpy.full(k, 2.0)
scl = _cabi.Scale(_cabi.SCALE_LINEAR, lo, hi)
traj = 2 * n * (1 + k)
vm = torch.empty(traj * L, dtype=torch.float64, device=dev)
ms_mid = kernel_ms(lambda: ctx.eval_values(k, n, p, _cabi.OBJ_MASS_ACTION, mid, scale=scl, out=vm))
finite = bool(torch.isfinite(vm).all())
del vm
ts = []
for _ in range(3):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    v = vb.Varsens(Packed(mid), lambda x: vb.linear(x, lo, hi), k, n, verbose=False)
    torch.cuda.synchronize()
    ts.append(time.perf_counter() - t0)
out["mid_network"] = {"S": S, "R": R, "L": L, "k": k, "n": n, "steps": steps, "trajectories": traj, "kernel_ms": ms_mid,
                      "trajectories_per_s": traj / (ms_mid * 1e-3), "values_finite": finite,
                      "varsens_end_to_end_s": min(ts), "sens_shape": list(v.sens.shape)}

# ---- 3. the same network through the @vectorized torch route, reduced n
net = ob.unpack(mid, adaptive=False)
rec, init = net.rec, net.init
W = torch.tensor(net.w, dtype=torch.float64, device=dev)
Nmat = torch.tensor(net.N, dtype=torch.float64, device=dev)
ix = {name: torch.tensor([int(q[c]) if q[c] >= 0 else S for q in rec], device=dev) for name, c in (("a0", 0), ("a1", 1), ("b0", 2), ("b1", 3))}
kfc = torch.tensor([int(q[4]) if q[4] >= 0 else k for q in rec], device=dev)
krc = torch.tensor([int(q[6]) if q[6] >= 0 else k for q in rec], device=dev)
kfv = torch.tensor([0.0 if q[4] >= 0 else q[5] for q in rec], dtype=torch.float64, device=dev)
krv = torch.tensor([0.0 if q[6] >= 0 else q[7] for q in rec], dtype=torch.float64, device=dev)
icc = torch.tensor([int(q[0]) if q[0] >= 0 else k for q in init], device=dev)
icv = torch.tensor([0.0 if q[0] >= 0 else q[1] for q in init], dtype=torch.float64, device=dev)


@vb.vectorized
def network_torch(P):                                            # (rows, k) -> (rows, L)
    rows = P.shape[0]
    pad = lambda A, v: torch.cat((A, v.expand(rows, -1)), dim=1)  # noqa: E731  (column k / S holds the constants)
    Pk = P
    kf = pad(Pk, torch.zeros(1, 1, dtype=P.dtype, device=P.device))[:, kfc] + kfv
    kr = pad(Pk, torch.zeros(1, 1, dtype=P.dtype, device=P.device))[:, krc] + krv
    X = pad(Pk, torch.zeros(1, 1, dtype=P.dtype, device=P.device))[:, icc] + icv
    one = torch.ones(1, 1, dtype=P.dtype, device=P.device)

    def rhs(Y):
        Yp = pad(Y, one)
        flux = kf * Yp[:, ix["a0"]] * Yp[:, ix["a1"]] - kr * Yp[:, ix["b0"]] * Yp[:, ix["b1"]]
        return flux @ Nmat.T

    h = 0.01
    for _ in range(steps):
        k1 = rhs(X)
        k2 = rhs(X + (0.5 * h) * k1)
        k3 = rhs(X + (0.5 * h) * k2)
        k4 = rhs(X + h * k3)
        X = X + (h / 6.0) * (k1 + 2.0 * k2 + 2.0 * k3 + k4)
    return X @ W.T


n_t = 1 << 10
ts = []
for _ in range(2):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    vt = vb.Varsens(network_torch, lambda x: vb.linear(x, lo, hi), k, n_t, verbose=False)
    torch.cuda.synchronize()
    ts.append(time.perf_counter() - t0)
vk = vb.Varsens(Packed(mid), lambda x: vb.linear(x, lo, hi), k, n_t, verbose=False)
traj_t = 2 * n_t * (1 + k)
out["torch_route"] = {"n": n_t, "trajectories": traj_t, "varsens_end_to_end_s": min(ts), "trajectories_per_s": traj_t / min(ts),
                      "max_abs_diff_sens_vs_kernel": float(numpy.abs(vt.sens - vk.sens).max())}
print(json.dumps(out, indent=1))
