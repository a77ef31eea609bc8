"""Multi-GPU plumbing for the hot path (SURVEY.md section 8e): one process per GPU, the independent odeint problems
of a training step (train_insilico.py:128-130) are sharded across ranks, the six weight tensors are replicated, and
the ONLY exchange is one sum-allreduce of the flat parameter-gradient vector per optimiser step (NCCL over
NVLink 5 / NVSwitch on the B200 box, gloo in the CPU tests).  The reference has no distributed code at all."""
import torch
import torch.distributed as dist

from . import engine


def shard_range(n_items, rank, world_size):
    """Contiguous, balanced slice [lo, hi) of n_items independent samples for this rank."""
    base, rem = divmod(n_items, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def flatten_grads(net):
    """The six .grad tensors concatenated in the reference parameter order (zeros where a grad is missing)."""
    parts = []
    for p in engine.net_params(net):
        g = p.grad if p.grad is not None else torch.zeros_like(p)
        parts.append(g.reshape(-1))
    return torch.cat(parts)


def flat_grad_view(net):
    """The six ``.grad`` tensors as ONE flat ``[P]`` tensor WITHOUT a copy, or None.  The adjoint kernels write the
    parameter cotangents into one flat buffer (reference order) and hand autograd six views of it; when a parameter has
    no gradient yet autograd keeps that view as ``.grad``, so after ``backward()`` the six gradients normally still sit
    back to back in one storage -- which is what lets the collective below run in place."""
    params = engine.net_params(net)
    g0 = params[0].grad
    if g0 is None:
        return None
    st, off = g0.untyped_storage(), g0.storage_offset()
    for p in params:
        g = p.grad
        if (g is None or g.dtype != g0.dtype or not g.is_contiguous() or g.storage_offset() != off
                or g.untyped_storage().data_ptr() != st.data_ptr()):
            return None
        off += g.numel()
    return torch.empty(0, dtype=g0.dtype, device=g0.device).set_(st, g0.storage_offset(), (off - g0.storage_offset(),))


def adopt_flat_grads_(net, flat, keep=None):
    """Make the six ``.grad`` tensors views of ``flat`` (no copy).  ``keep``: six flags; a parameter whose flag is False
    keeps ``.grad`` None (a parameter outside the adjoint set got no gradient, and an optimiser must not move it)."""
    o = 0
    for i, p in enumerate(engine.net_params(net)):
        n = p.numel()
        if keep is None or keep[i]:
            p.grad = flat[o:o + n].view_as(p)
        o += n


def unflatten_grads_(net, flat):
    o = 0
    for p in engine.net_params(net):
        n = p.numel()
        if p.grad is None:
            p.grad = flat[o:o + n].view_as(p).clone()
        else:
            p.grad.copy_(flat[o:o + n].view_as(p))
        o += n


def allreduce_grads(net, group=None, average=True, extra=None):
    """Combine the parameter gradients (and optional extra scalars such as the loss) of all ranks.

    ``average=True`` (default) divides the sum by the world size: the reference's losses are ``torch.mean`` over the
    LOCAL samples (train_insilico.py:132,135), so with the samples of a step sharded over the ranks the averaged gradient
    is the single-GPU gradient (exactly when the shards are equal, up to the shard-size weighting otherwise) and the
    learning rate keeps its meaning as N grows.  A caller that normalises its losses by the GLOBAL batch size itself
    (tools/train_epoch.py) passes ``average=False`` to get the plain sum.

    One collective over the flat ``[P]`` gradient, IN PLACE when the six gradients are views of one buffer
    (``flat_grad_view``: the normal case after a backward through this package -- no gather / scatter passes over the
    35.8 MB vector); otherwise they are gathered once and ``.grad`` becomes views of the reduced buffer (no copy back).
    ``extra`` rides in a second, tiny collective in the first case and at the tail of the vector in the second.
    A parameter without a gradient (frozen, or left out of ``adjoint_params``; the same on every rank) enters the sum as
    zeros and keeps ``.grad`` None."""
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return extra
    world = dist.get_world_size(group)
    pr = _peer.get(id(net))
    if pr is not None:
        return _peer_allreduce_grads(net, pr, average, extra)
    flat = flat_grad_view(net)
    if flat is not None:
        work = dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group, async_op=extra is not None)
        out = None
        if extra is not None:
            out = extra.reshape(-1).to(flat.dtype).clone()
            dist.all_reduce(out, op=dist.ReduceOp.SUM, group=group)
            work.wait()
            out = out.view_as(extra)
        if average:
            flat /= world
            if out is not None:
                out /= world
        return out
    had = [p.grad is not None for p in engine.net_params(net)]
    flat = flatten_grads(net)
    n = flat.numel()
    if extra is not None:
        flat = torch.cat([flat, extra.reshape(-1).to(flat.dtype)])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    if average:
        flat /= world
    adopt_flat_grads_(net, flat[:n], had)
    return flat[n:].view_as(extra) if extra is not None else None


# ---- gradient all-reduce over peer memory (csrc/phx_peer.cu) -----------------------------------------------------------------
class PeerAllReduce:
    """In-place sum of a flat float32 vector over the GPUs of one NVSwitch box through peer memory: ONE kernel per rank
    (``phx_peer_allreduce``: reduce-scatter by slices with remote loads, all-gather with remote stores, rank-ordered sums,
    bit-identical results on every rank), no NCCL call on the data path.  torch symmetric memory only provides the
    peer-mapped allocation and the pointer exchange.  ``buffer`` is this rank's vector (``numel`` floats): write the local
    gradient into it, call ``reduce()``; afterwards it holds ``scale * sum``."""

    def __init__(self, numel, device=None, group=None, nvls=None):
        import torch.distributed._symmetric_memory as symm_mem
        from . import _lib
        self.group = dist.group.WORLD if group is None else group
        self.world, self.rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        if self.world not in (2, 4, 8):
            raise NotImplementedError("peer all-reduce: 2, 4 or 8 ranks (got %d)" % self.world)
        self.dev = torch.cuda.current_device() if device is None else torch.device(device).index
        d = torch.device("cuda", self.dev)
        self.numel = int(numel)
        self.buffer = symm_mem.empty((self.numel + 3) // 4 * 4, dtype=torch.float32, device=d)
        self.flags = symm_mem.empty(64, dtype=torch.int32, device=d)
        self.flags.zero_()
        self.buffer.zero_()
        hb = symm_mem.rendezvous(self.buffer, self.group)
        hf = symm_mem.rendezvous(self.flags, self.group)
        import ctypes
        self._bufs = (ctypes.c_void_p * self.world)(*[int(x) for x in hb.buffer_ptrs])
        self._flags = (ctypes.c_void_p * self.world)(*[int(x) for x in hf.buffer_ptrs])
        self._handles = (hb, hf)
        # NVLS (sums formed inside the NVSwitch, phx_peer_allreduce_nvls) when the buffer has a multicast address:
        # nvls=None -> PHX_PEER_NVLS (default: on at 8 ranks -- measured for the 35.8 MB gradient: 4 GPUs 105 us peer
        # loads / stores vs 127 us NVLS, 8 GPUs 147 vs 134 us), True / False force it
        try:
            self._mc = int(hb.multicast_ptr or 0)
        except Exception:   # no multicast support on this box / torch build
            self._mc = 0
        if nvls is None:
            import os
            env = os.environ.get("PHX_PEER_NVLS")
            nvls = (self.world >= 8) if env is None else bool(int(env))
        self.nvls = bool(nvls) and self._mc != 0
        self.epoch = 0
        self._lib, self._ctx = _lib.load(), _lib.ctx(self.dev)
        self._check = _lib.check
        torch.cuda.synchronize(d)
        dist.barrier(group=self.group)      # every rank's flag pad is zero before anyone signals

    def reduce(self, scale=1.0, numel=None):
        self.epoch += 1
        n = self.numel if numel is None else int(numel)
        if self.nvls:
            self._check(self._lib.phx_peer_allreduce_nvls(self._ctx, self._mc, self._flags, self.rank, self.world, n,
                                                          self.epoch & 0x7fffffff, float(scale),
                                                          engine._stream_ptr(self.dev)), "peer_allreduce_nvls")
        else:
            self._check(self._lib.phx_peer_allreduce(self._ctx, self._bufs, self._flags, self.rank, self.world, n,
                                                     self.epoch & 0x7fffffff, float(scale),
                                                     engine._stream_ptr(self.dev)), "peer_allreduce")
        return self.buffer[:n]


_peer = {}


def enable_peer_allreduce(net, group=None):
    """Route ``allreduce_grads(net)`` through ``PeerAllReduce`` (one peer-memory kernel instead of an NCCL all-reduce).
    Collective: call on every rank.  Returns the PeerAllReduce object (``.buffer`` can be written directly)."""
    params = engine.net_params(net)
    P = sum(p.numel() for p in params)
    pr = PeerAllReduce(P + 64, device=params[0].device, group=group)     # 64 spare floats for the `extra` scalars
    _peer[id(net)] = pr
    base = pr.buffer.untyped_storage().data_ptr()

    def alloc(n):
        # the adjoint kernels write the flat gradient straight into the peer-mapped buffer -- unless a .grad of an earlier
        # backward still lives there (gradient accumulation over several backward calls)
        for p in params:
            if p.grad is not None and p.grad.untyped_storage().data_ptr() == base:
                return None
        return pr.buffer[:n] if n == P else None

    engine._flat_alloc[id(net)] = alloc
    return pr


def try_enable_peer_allreduce(net, group=None):
    """``enable_peer_allreduce`` that falls back to NCCL (returns None) when peer-mapped memory cannot be set up on this
    box / torch build.  The ranks agree on the outcome (a failure on one rank disables it everywhere)."""
    import sys
    dev = engine.net_params(net)[0].device

    def agree(ok):
        flag = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
        return int(flag) == 1

    pr, err = None, None
    try:
        pr = enable_peer_allreduce(net, group=group)
    except Exception as e:   # noqa: BLE001 -- any set-up failure means "use NCCL"
        err = e
    ok = agree(pr is not None)          # before the first kernel: a rank without buffers must not leave the others spinning
    if ok:
        try:
            pr.buffer[:4].fill_(1.0)
            pr.reduce(numel=4)
            torch.cuda.synchronize()
            ok = abs(float(pr.buffer[0]) - pr.world) < 1e-3
        except Exception as e:   # noqa: BLE001
            ok, err = False, e
        ok = agree(ok)
    if ok:
        return pr
    disable_peer_allreduce(net)
    if dist.get_rank(group) == 0:
        sys.stderr.write("phoenix_b200: peer-memory all-reduce unavailable (%s); using NCCL\n" % (err,))
    return None


def disable_peer_allreduce(net):
    _peer.pop(id(net), None)
    engine._flat_alloc.pop(id(net), None)


def _peer_allreduce_grads(net, pr, average, extra):
    params = engine.net_params(net)
    P = sum(p.numel() for p in params)
    flat = flat_grad_view(net)
    had = [p.grad is not None for p in params]
    buf = pr.buffer
    in_place = flat is not None and flat.data_ptr() == buf.data_ptr()
    if not in_place:
        if flat is not None:
            buf[:P].copy_(flat)
        else:   # gradients in several storages (some may already sit at their place in the peer buffer)
            o = 0
            for p in params:
                k = p.numel()
                if p.grad is None:
                    buf[o:o + k].zero_()
                elif p.grad.data_ptr() != buf.data_ptr() + 4 * o:
                    buf[o:o + k].copy_(p.grad.reshape(-1))
                o += k
    n = P
    if extra is not None:
        if extra.numel() > 64:
            raise ValueError("allreduce_grads: at most 64 extra scalars ride with the gradient")
        buf[P:P + extra.numel()].copy_(extra.reshape(-1))
        n = P + extra.numel()
    pr.reduce(scale=(1.0 / pr.world) if average else 1.0, numel=n)
    if not in_place:
        adopt_flat_grads_(net, buf[:P], had)
    return buf[P:n].clone().view_as(extra) if extra is not None else None


def broadcast_parameters(net, src=0, group=None):
    """Replicate rank `src`'s six weight tensors on every rank (start of training / after loading a checkpoint)."""
    if not dist.is_available() or not dist.is_initialized():
        return
    with torch.no_grad():
        for p in engine.net_params(net):
            dist.broadcast(p, src=src, group=group)
    engine.invalidate(net)   # the collective writes the storages without bumping the version counters


# ---- exact global error norm for a batched dopri5 solve sharded over ranks (SURVEY 8e caveat) -------------------------------
_SUM_HOOK_T = None
_sum_hooks = {}


class _DeviceDoubles:
    """A raw device pointer to n float64 values as a CUDA-array-interface object (torch.as_tensor wraps it, no copy)."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 2}


def enable_global_norm(device=None, group=None):
    """A single batched ``odeint`` call uses ONE error norm over all its rows (torchdiffeq/_impl/misc.py:10-11).  When the
    rows of such a call are split over ranks, call this once per rank (same number of rows on every rank): every norm
    evaluation of the streaming dopri5 forward solve then all-reduces its partial sums (3 doubles) over `group`, so all
    ranks take identical accept / reject decisions -- the same step sequence as the unsharded call, up to summation
    order.  Without it each rank steps by the norm of its own shard.  ``disable_global_norm`` switches it off."""
    import ctypes
    global _SUM_HOOK_T
    from . import _lib
    if not dist.is_available() or not dist.is_initialized():
        return
    dev = torch.cuda.current_device() if device is None else torch.device(device).index
    if _SUM_HOOK_T is None:
        _SUM_HOOK_T = ctypes.CFUNCTYPE(None, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p)

    def hook(ptr, n, stream, user):
        t = torch.as_tensor(_DeviceDoubles(ptr, n), device=torch.device("cuda", dev))
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)

    cb = _SUM_HOOK_T(hook)
    _sum_hooks[dev] = cb          # keep the trampoline alive
    _lib.check(_lib.load().phx_ctx_set_global_norm(_lib.ctx(dev), ctypes.cast(cb, ctypes.c_void_p), None,
                                                   dist.get_world_size(group)), "set_global_norm")


def disable_global_norm(device=None):
    from . import _lib
    dev = torch.cuda.current_device() if device is None else torch.device(device).index
    _lib.check(_lib.load().phx_ctx_set_global_norm(_lib.ctx(dev), None, None, 1), "set_global_norm")
    _sum_hooks.pop(dev, None)
