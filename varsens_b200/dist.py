"""Multi-GPU plumbing: one process per GPU (torch.distributed, NCCL over NVLink), base rows sharded
over ranks, ONE all-reduce of the O(k^2) partial-sum vector (SURVEY.md §8e).  The reference's only
scale-out mechanism is file batching (varsens/saltelli.py:173-193 -> cluster/accre-submit.sh:27 ->
:415-472); this replaces it for registered functors.  Export mode needs no collective at all:
every rank writes its own contiguous window of flat rows."""
import os

from ._cabi import objective_outputs


def world():
    """(rank, world_size) of the initialised torch.distributed process group, else (0, 1).

    The torchrun environment (RANK / WORLD_SIZE) alone is NOT enough: rows are only sharded when a reduction over the
    same group is guaranteed to follow.  Under torchrun without ``init_process_group`` every process therefore runs the
    whole design (correct, merely redundant) instead of finalising its own shard's sums as if they were the total."""
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist.get_rank(), dist.get_world_size()
    except ImportError:
        pass
    return 0, 1


def shard_range(total, rank, world_size):
    """Contiguous slice [lo, hi) of `total` units owned by `rank`; sizes differ by at most one."""
    total, rank, world_size = int(total), int(rank), int(world_size)
    if not 0 <= rank < world_size:
        raise ValueError("rank %d outside world of %d" % (rank, world_size))
    base, extra = divmod(total, world_size)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def allreduce_partials(partials, group=None):
    """In-place SUM all-reduce of a rank's partial-sum tensor (fp64; ~10 KB at k=20).  `partials` is a
    torch tensor on this rank's device (cuda -> NCCL, cpu -> gloo).  Enqueued on torch's current stream: run the ctx on
    that stream (on_torch_stream) so that the producing kernel and the finalisation are ordered around it."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(partials, op=dist.ReduceOp.SUM, group=group)
    return partials


def partials_layout(k, l=1):
    """Index helpers for the partial-sum vector (include/varsens_b200.h: vs_partials_len)."""
    m = (2 + 2 * k) * l

    def gram(p, q):
        if p > q:
            p, q = q, p
        return 4 * l + p * m - p * (p - 1) // 2 + (q - p)

    return dict(m=m, length=4 * l + m * (m + 1) // 2, S_A=0, S_B=l, Q_A=2 * l, Q_B=3 * l, gram=gram)


class PeerExchange(object):
    """Exchange buffers of the peer-memory all-reduce (vs_run_fused_p2p, vs_allreduce_finalize_p2p): one torch symmetric-memory
    allocation per rank, mapped into every process of the group over NVLink.  Layout per rank: 2 sets (epoch parity) x world
    slots x plen elements x 16 bytes -- every double travels as {lo, epoch, hi, epoch} (include/varsens_b200.h) -- zeroed."""

    def __init__(self, plen, device, group=None):
        import torch
        import torch.distributed as tdist
        import torch.distributed._symmetric_memory as symm
        self.group = tdist.group.WORLD if group is None else group
        self.world = tdist.get_world_size(self.group)
        self.rank = tdist.get_rank(self.group)
        self.plen = int(plen)
        nslots = 2 * self.world * self.plen
        self.buf = symm.empty(2 * nslots + 16, dtype=torch.float64, device=device)
        self.buf.zero_()
        self.handle = symm.rendezvous(self.buf, self.group)
        base = [int(p_) for p_ in self.handle.buffer_ptrs]
        self.peer_bufs = base
        self.peer_flags = base                        # the low-latency protocol tags every element; no separate flag array
        self.epoch = 0
        torch.cuda.synchronize(device)
        tdist.barrier(self.group)                     # every rank's buffer is zeroed before anybody stores into it

    def next_epoch(self):
        self.epoch += 1
        return self.epoch


_exchanges = {}


def peer_exchange(plen, device, group=None):
    """Cached PeerExchange for (plen, device); None if symmetric memory is not available (then use NCCL)."""
    key = (int(plen), str(device))
    if key not in _exchanges:
        try:
            _exchanges[key] = PeerExchange(plen, device, group)
        except Exception as exc:                      # no NVLink peer access / no symmetric-memory support
            if os.environ.get("VS_P2P_STRICT"):
                raise
            _exchanges[key] = None
            print("varsens_b200: peer-memory all-reduce unavailable (%s); using NCCL" % (exc,))
    return _exchanges[key]


def use_nccl():
    """VS_NCCL=1 selects the NCCL all-reduce (+ finalize kernel) instead of the one-launch peer-memory step."""
    return os.environ.get("VS_NCCL", "0") == "1"


def outputs_of_partials(k, length):
    """The outputs per point l whose partial-sum vector for k factors has `length` entries."""
    for l in range(1, 65):
        if partials_layout(k, l)["length"] == int(length):
            return l
    raise ValueError("%d is not a partial-sum length for k = %d" % (length, k))


def reduce_and_finalize(ctx, k, n, part, flags):
    """Sum a rank's partial-sum tensor over the group and compute the indices (every rank returns the same Result; the
    outputs per point l follow from the tensor's length).
    Default: the stand-alone peer-memory exchange kernel (vs_allreduce_finalize_p2p) over torch symmetric memory; with
    VS_NCCL=1, or when symmetric memory is unavailable: one NCCL all_reduce followed by vs_finalize.  The collective runs
    on torch's current stream, so the ctx is switched onto that stream for the call: the kernel that produced `part`,
    the all-reduce and the finalisation are then ordered by the stream itself."""
    import torch
    rank, ws = world()
    l = outputs_of_partials(k, part.numel())
    if ws == 1:
        return ctx.finalize(k, l, n, part, flags)
    ex = None if use_nccl() else peer_exchange(part.numel(), part.device)
    with on_torch_stream(ctx, part.device):
        if ex is not None:
            return ctx.allreduce_finalize_p2p(k, l, n, ex.world, ex.rank, ex.peer_bufs, ex.peer_flags, ex.next_epoch(), part, flags)
        allreduce_partials(part)
        return ctx.finalize(k, l, n, part, flags)


class on_torch_stream(object):
    """Run a ctx on torch's current stream for the duration of a block (vs_ctx_set_stream synchronises the stream it
    leaves, so work enqueued before and after is ordered too); restores the ctx's own stream afterwards."""

    def __init__(self, ctx, device):
        self.ctx, self.device = ctx, device

    def __enter__(self):
        import torch
        self.prev = getattr(self.ctx, "_stream_ptr", None)
        self.ctx.set_stream(torch.cuda.current_stream(self.device).cuda_stream)
        return self.ctx

    def __exit__(self, *exc):
        self.ctx.set_stream(self.prev)
        return False


def fused_step(ctx, k, n, perm, objective, params, discard, scale, raw, flags):
    """The fused Saltelli step over the whole process group: this rank evaluates its contiguous shard of the n base rows
    and every rank returns the indices of the full design.

    Default (NVLink peer memory available): ONE kernel launch per rank -- vs_run_fused_p2p: generation, evaluation, Gram,
    the all-reduce of the partial sums over peer memory and the estimators, results in mapped host memory.
    VS_NCCL=1 (or no symmetric memory): vs_fused_partials -> one NCCL all_reduce -> vs_finalize."""
    import torch
    rank, ws = world()
    if ws == 1:
        return ctx.run_fused(k, n, perm, objective, params, discard, scale, raw, flags)
    lo, hi = shard_range(n, rank, ws)
    device = torch.device("cuda", ctx.device)
    l = objective_outputs(k, objective, params)
    plen = partials_layout(k, l)["length"]
    ex = None if use_nccl() else peer_exchange(plen, device)
    if ex is not None and hi > lo:
        return ctx.fused_plan(k, n, perm, objective, params, discard, scale, raw, flags, lo, hi, ex).run()
    part = torch.empty(plen, dtype=torch.float64, device=device)
    with on_torch_stream(ctx, device):
        ctx.fused_partials(k, n, perm, objective, params, discard, scale, raw, lo, hi, flags, out=part)
        allreduce_partials(part)
        return ctx.finalize(k, l, n, part, flags)
