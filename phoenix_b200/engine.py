"""Host-side glue between torch tensors and the C ABI: packed-weight cache, workspaces, status records.

PyTorch is used here only as the owner of device memory and streams; every kernel lives in libphoenix_b200.so.
"""
import ctypes
import threading
import weakref

import torch

from . import _lib

# solver "assert" conditions (rk_common.py:154,175-176) are checked when the status record is read.  With
# SYNC_ERRORS (the default: exact reference behaviour) the stream is synchronised after every solve and the reference's
# AssertionError is raised at the call site.  set_sync_errors(False) is an explicit opt-in to lazy checking, which keeps
# the host running ahead of the GPU (a loop of per-sample calls pipelines): the records are then inspected at the start
# of every later solve, by check_errors(), and at interpreter exit; outputs a failed solve did not reach are NaN.
SYNC_ERRORS = True
STEP_LOGGING = False
STEPLOG_CAP = 4096
FORCE_ENGINE = None  # None | "rows" | "resident" | "stream"  (tests compare the engines on the same inputs)
# A ONE-sample odeint / odeint_adjoint call (the literal loop of train_insilico.py:128-130) on a model whose solve fills the
# GPU: "resident" = the one-problem persistent kernels (forward 79 us + backward 370 us per call at 11 165 x 200, flat
# gradient written directly), "rows" = the lock-step rows kernels with a single row (107 + 425 us: a pass costs the same
# with 1 row as with 4, plus the packed -> flat conversion) -- bit-identical to odeint_adjoint_many, which always uses them.
SINGLE_CALL_ENGINE = "resident"
SINGLE_CALL_MIN_GENES = 2048

class _State:
    """Process-wide bookkeeping (NOT thread-local: autograd runs backward() on its own worker thread)."""

    def __init__(self):
        self.lock = threading.RLock()
        self.pending = []       # [(status_tensor, what)]
        self.free_status = []
        self.last_log = None
        self.last_status = None
        self.last_status_block = None
        self.workspaces = {}


_state = _State()
_last_rhs = {}   # rhs workspace data_ptr -> signature of the phx_rhs_forward call whose [S|P] it still holds


def set_sync_errors(flag):
    global SYNC_ERRORS
    SYNC_ERRORS = bool(flag)


def _report_pending_at_exit():
    try:
        check_errors()
    except AssertionError as exc:   # lazy mode only: a failed solve nobody asked about
        import sys
        sys.stderr.write("phoenix_b200: a solve hit a solver assertion that was never checked: %s\n" % exc)
    except Exception:
        pass


import atexit  # noqa: E402
atexit.register(_report_pending_at_exit)


def set_step_logging(flag):
    """Record (t0, dt, accepted) for every attempted adaptive step of subsequent solves (tests / diagnostics)."""
    global STEP_LOGGING
    STEP_LOGGING = bool(flag)


_PRECISIONS = {"fp32": _lib.PREC_FP32, "tf32": _lib.PREC_TF32, "3xtf32": _lib.PREC_3XTF32}


def set_precision(mode, device=None):
    """Arithmetic of the dense (B >= 5 rows) contractions: '3xtf32' (default; tcgen05 tensor cores with the
    three-term TF32 split, fp32 parity), 'tf32' (single-pass TF32, ~1e-3 relative error) or 'fp32' (CUDA cores).
    Smaller batches are GEMV-bound and always run in fp32 on the CUDA cores."""
    if mode not in _PRECISIONS:
        raise ValueError("precision must be one of %s" % sorted(_PRECISIONS))
    dev = torch.cuda.current_device() if device is None else torch.device(device).index
    _lib.check(_lib.load().phx_ctx_set_precision(_lib.ctx(dev), _PRECISIONS[mode]), "set_precision")


def _tls():
    return _state


def _device_index(t):
    if not t.is_cuda:
        raise RuntimeError(
            "phoenix_b200 runs the PHOENIX hot path on a B200 only: got a tensor on %s. Move the model and its inputs "
            "to 'cuda' (there is no CPU fallback)." % t.device)
    return t.device.index if t.device.index is not None else torch.cuda.current_device()


def _stream_ptr(dev):
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _workspace(dev, nbytes, tag):
    tls = _tls()
    key = (dev, tag, torch.cuda.current_stream(dev).cuda_stream)
    ws = tls.workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=torch.device("cuda", dev))
        if tag == "rhs":
            _last_rhs.clear()   # a new buffer holds nothing (and a freed one may come back at the same address)
        if tag == "solve":
            # the resident solvers keep their inter-CTA exchange area at the start of the workspace: zero it once
            lib = _lib.load()
            _lib.check(lib.phx_solve_workspace_init(_ptr(ws), ws.numel(), _stream_ptr(dev)), "workspace_init")
        tls.workspaces[key] = ws
    return ws


# ---- packed weights ------------------------------------------------------------------------------------------------
def _lin(net, name):
    # nn.Module keeps parameters / submodules in dicts and only reaches them through the slow __getattr__ fallback;
    # this runs twice per sample of every training step, so go to the dicts directly
    return net._modules[name]._modules["linear_out"]._parameters


def net_params(net):
    """The six parameters in the reference's ``ODENet.parameters()`` order (adjoint.py:185,207-220)."""
    prods, sums = _lin(net, "net_prods"), _lin(net, "net_sums")
    return [net._parameters["gene_multipliers"], prods["weight"], prods["bias"], sums["weight"], sums["bias"],
            _lin(net, "net_alpha_combine")["weight"]]


def net_dims(net):
    W = _lin(net, "net_sums")["weight"]
    return int(W.shape[1]), int(W.shape[0])


_pack_cache = weakref.WeakKeyDictionary()


def _on_model_device(fn):
    """Run an entry point with the model's device current (the caller may sit on another GPU): launches, workspaces
    and streams all follow torch's current device."""
    import functools

    @functools.wraps(fn)
    def wrapper(net, *args, **kwargs):
        p0 = net._parameters["gene_multipliers"]
        if p0.is_cuda and p0.device.index != torch.cuda.current_device():
            with torch.cuda.device(p0.device):
                return fn(net, *args, **kwargs)
        return fn(net, *args, **kwargs)
    return wrapper


@_on_model_device
def packed_weights(net):
    """Kernel-layout copy of the parameters, rebuilt only when a parameter changed (``_version`` / storage)."""
    params = net_params(net)
    ent = _pack_cache.get(net)
    if ent is not None:
        # fast path (every call between two optimiser steps): same storages, same versions, same stream
        dev = ent[3]
        key = tuple((p.data_ptr(), p._version) for p in params) + (torch.cuda.current_stream(dev).cuda_stream,)
        if ent[0] == key:
            return ent[1], ent[2][0], ent[2][1], dev
    G, H = net_dims(net)
    dev = _device_index(params[0])
    for p in params:
        if p.dtype != torch.float32:
            raise TypeError("phoenix_b200 computes in float32; parameter has dtype %s (call odenet.float())" % p.dtype)
        if _device_index(p) != dev:
            raise RuntimeError("all ODENet parameters must live on the same CUDA device")
    key = tuple((p.data_ptr(), p._version) for p in params) + (torch.cuda.current_stream(dev).cuda_stream,)
    lib = _lib.load()
    nbytes = lib.phx_packed_bytes(G, H)
    buf = ent[1] if ent is not None and ent[1].numel() * 4 == nbytes and ent[1].device.index == dev else \
        torch.empty(nbytes // 4, dtype=torch.float32, device=torch.device("cuda", dev))
    ps = [p.detach().contiguous() for p in params]
    _lib.check(lib.phx_pack_weights(_lib.ctx(dev), G, H, *[_ptr(p) for p in ps], _ptr(buf), _stream_ptr(dev)),
               "pack_weights")
    _pack_cache[net] = (key, buf, (G, H), dev)
    return buf, G, H, dev


def invalidate(net=None):
    """Drop the cached kernel-layout copy of `net`'s parameters (all models if None).  The cache is keyed on each
    parameter's storage pointer and autograd version counter; edits that bypass the counter -- ``p.data.mul_()``,
    ``torch.distributed.broadcast(p)`` under no_grad, writes through a raw pointer -- must be followed by a call to this
    function (``parallel.broadcast_parameters`` does it), otherwise the kernels keep integrating the old weights."""
    if net is None:
        for k in list(_pack_cache.keys()):
            del _pack_cache[k]
    elif net in _pack_cache:
        del _pack_cache[net]
    with _state.lock:
        _last_rhs.clear()


# ---- status records -----------------------------------------------------------------------------------------------------
def _poll_pending():
    """Lazy mode: raise for any solve that has already finished with a solver assertion (no synchronisation)."""
    if not SYNC_ERRORS and _tls().pending:
        check_errors(synchronize=False)


def _new_status():
    tls = _tls()
    _poll_pending()
    if tls.free_status:
        st = tls.free_status.pop()
    else:
        st = torch.empty(ctypes.sizeof(_lib.PhxStatus) // 4, dtype=torch.int32).pin_memory()
    # reset through ctypes (no torch dispatch on the per-sample path)
    ctypes.memset(st.data_ptr(), 0, ctypes.sizeof(_lib.PhxStatus))
    _lib.PhxStatus.from_address(st.data_ptr()).code = _lib.ST_RUNNING
    return st


def _status_struct(st):
    return _lib.PhxStatus.from_address(st.data_ptr())


def _raise_for(st, what):
    s = _status_struct(st)
    if s.code == _lib.ST_DT_UNDERFLOW:
        raise AssertionError("underflow in dt {}".format(s.dt_fail))
    if s.code == _lib.ST_NONFINITE:
        raise AssertionError("non-finite values in state `y` ({}, t={})".format(what, s.t_fail))
    if s.code == _lib.ST_MAX_STEPS:
        raise AssertionError("max_num_steps exceeded ({}, t={})".format(what, s.t_fail))


def check_errors(synchronize=True):
    """Raise the reference's AssertionError for any finished solve that hit a solver assertion."""
    tls = _tls()
    if synchronize and torch.cuda.is_available():
        torch.cuda.synchronize()
    still = []
    err = None
    for st, what in tls.pending:
        code = _status_struct(st).code
        if code == _lib.ST_RUNNING:
            still.append((st, what))
            continue
        if code != _lib.ST_OK and err is None:
            err = (st, what)
        else:
            tls.free_status.append(st)
    tls.pending = still
    if err is not None:
        _raise_for(*err)


def last_step_log(problem=None):
    """(t0, dt, accepted) rows of the most recent solve (requires set_step_logging(True)); synchronises.  After a
    multi-problem call ``problem`` selects the sample (default: the last one, like a loop of single calls would leave)."""
    tls = _tls()
    if tls.last_log is None:
        return []
    torch.cuda.synchronize()
    log = tls.last_log
    if log.dim() == 3:
        i = log.shape[0] - 1 if problem is None else problem
        n = _status_struct(tls.last_status_block[i]).n_logged
        return [tuple(r) for r in log[i, :n].tolist()]
    n = _status_struct(tls.last_status).n_logged
    return [tuple(r) for r in log[:n].tolist()]


def last_status():
    tls = _tls()
    if tls.last_status is None:
        return None
    torch.cuda.synchronize()
    s = _status_struct(tls.last_status)
    return {"code": s.code, "n_accepted": s.n_accepted, "n_rejected": s.n_rejected, "n_rhs": s.n_rhs,
            "n_logged": s.n_logged}


def _finish(st, what, dev):
    tls = _tls()
    tls.last_status = st
    if SYNC_ERRORS:
        torch.cuda.current_stream(dev).synchronize()
        code = _status_struct(st).code
        if code != _lib.ST_OK:
            _raise_for(st, what)
        tls.free_status.append(st)
    else:
        tls.pending.append((st, what))
        if len(tls.pending) > 64:
            check_errors(synchronize=False)


def _steplog():
    tls = _tls()
    if not STEP_LOGGING:
        tls.last_log = None
        return None, 0
    log = torch.zeros(STEPLOG_CAP, 3, dtype=torch.float64).pin_memory()
    tls.last_log = log
    return log, STEPLOG_CAP


# ---- cached Hill activations of constant inputs (csrc/phx_tc.cu, "cached Hill activations") ------------------------------
# (data_ptr, numel) -> (weakref to the caller's tensor, its version, s plane, l plane)
_hill_planes = {}
_hill_seen = {}
CACHE_ACTIVATIONS = True   # 2 x the size of the cached input in HBM (0.9 GB for the 10 000 x 11 165 prior batch)


def hill_planes_for(x2, src, dev):
    """s(x), l(x) planes of x2 (contiguous fp32 view of the caller's tensor `src`), cached while `src` is alive and
    unmodified; None when caching is off or x2 is a converted copy."""
    import weakref
    if not CACHE_ACTIVATIONS or x2.data_ptr() != src.data_ptr():
        return None
    key = (x2.data_ptr(), x2.numel())
    ent = _hill_planes.get(key)
    if ent is not None and ent[0]() is src and ent[1] == src._version:
        return ent[2], ent[3]
    for k in [k for k, v in _hill_planes.items() if v[0]() is None]:   # the owner is gone: drop its planes
        del _hill_planes[k]
    lib = _lib.load()
    sp, lp = torch.empty_like(x2), torch.empty_like(x2)
    _lib.check(lib.phx_hill_planes(_lib.ctx(dev), x2.numel(), _ptr(x2), _ptr(sp), _ptr(lp), _stream_ptr(dev)),
               "hill_planes")
    _hill_planes[key] = (weakref.ref(src), src._version, sp, lp)
    return sp, lp


def _auto_hill_planes(x2, src, dev):
    """prior_only_forward is only ever fed the constant prior batch (train_insilico.py:134): the second time the same
    unmodified tensor comes by, its activations are cached (the first sighting only leaves a note)."""
    import weakref
    if not CACHE_ACTIVATIONS or x2.data_ptr() != src.data_ptr():
        return None
    key = (x2.data_ptr(), x2.numel())
    ent = _hill_planes.get(key)
    if ent is not None and ent[0]() is src and ent[1] == src._version:
        return ent[2], ent[3]
    seen = _hill_seen.get(key)
    if seen is not None and seen[0]() is src and seen[1] == src._version:
        return hill_planes_for(x2, src, dev)
    if len(_hill_seen) > 64:
        _hill_seen.clear()
    _hill_seen[key] = (weakref.ref(src), src._version)
    return None


class hill_cache:
    """Scope in which the library reads cached planes for the contractions over x2.  The entry is set right before and
    cleared right after the launches: a stale one would silently feed another tensor allocated at the same address."""

    def __init__(self, dev, x2, planes):
        self.dev, self.x2, self.planes = dev, x2, planes

    def __enter__(self):
        if self.planes is not None:
            _lib.load().phx_hill_cache_set(_lib.ctx(self.dev), _ptr(self.x2), self.x2.numel(), _ptr(self.planes[0]),
                                           _ptr(self.planes[1]))

    def __exit__(self, *exc):
        if self.planes is not None:
            _lib.load().phx_hill_cache_set(_lib.ctx(self.dev), None, 0, None, None)
        return False


# ---- RHS -----------------------------------------------------------------------------------------------------------------
def _rhs_signature(net, packed, y2, B):
    key = _pack_cache.get(net)
    prec = _lib.load().phx_ctx_get_precision(_lib.ctx(_device_index(y2)))
    return (packed.data_ptr(), key[0] if key is not None else None, y2.data_ptr(), y2._version, tuple(y2.shape), B,
            prec)


@_on_model_device
def rhs_forward(net, y, decay):
    packed, G, H, dev = packed_weights(net)
    if y.shape[-1] != G:
        raise RuntimeError("last dimension of y (%d) must equal ndim (%d)" % (y.shape[-1], G))
    y2 = y.detach().to(torch.float32).contiguous()
    B = y2.numel() // G
    lib = _lib.load()
    f = torch.empty_like(y2)
    nb = lib.phx_rhs_workspace_bytes(G, H, B)
    ws = _workspace(dev, nb, "rhs")
    planes = _auto_hill_planes(y2, y, dev) if (not decay and B >= lib.phx_tc_min_rows()) else None
    with hill_cache(dev, y2, planes):
        _lib.check(lib.phx_rhs_forward(_lib.ctx(dev), G, H, B, _ptr(packed), _ptr(y2), _ptr(f), int(decay), _ptr(ws),
                                       ws.numel(), _stream_ptr(dev)), "rhs_forward")
    with _state.lock:
        _last_rhs[ws.data_ptr()] = _rhs_signature(net, packed, y2, B)
    return f


@_on_model_device
def rhs_vjp(net, y, g, decay, need_ybar=True, need_grads=True, flat=False):
    packed, G, H, dev = packed_weights(net)
    y2 = y.detach().to(torch.float32).contiguous()
    g2 = g.detach().to(torch.float32).contiguous()
    B = y2.numel() // G
    lib = _lib.load()
    ybar = torch.empty_like(y2) if need_ybar else None
    P = 4 * G * H + 2 * H + G
    grads = torch.empty(P, dtype=torch.float32, device=y2.device) if need_grads else None
    nb = lib.phx_rhs_workspace_bytes(G, H, B)
    ws = _workspace(dev, nb, "rhs")
    # the workspace still holds [S|P] of the forward call on exactly these weights and this y (training_step: prior
    # forward, then composed_loss.backward()): tell the library not to recompute it
    with _state.lock:
        reuse = _last_rhs.pop(ws.data_ptr(), None) == _rhs_signature(net, packed, y2, B)
    ent = _hill_planes.get((y2.data_ptr(), y2.numel())) if (not decay and CACHE_ACTIVATIONS) else None
    planes = (ent[2], ent[3]) if (ent is not None and ent[0]() is not None and ent[1] == y._version
                                  and y2.data_ptr() == y.data_ptr()) else None
    with hill_cache(dev, y2, planes):
        _lib.check(lib.phx_rhs_vjp(_lib.ctx(dev), G, H, B, _ptr(packed), _ptr(y2), _ptr(g2), int(decay), _ptr(ybar),
                                   _ptr(grads), 2 if reuse else 0, _ptr(ws), ws.numel(), _stream_ptr(dev)), "rhs_vjp")
    if flat:   # the caller scales / splits the [P] vector itself
        return ybar, grads
    return ybar, (split_flat_grads(grads, G, H) if need_grads else None)


# net id -> callable(P) returning a [P] float32 tensor on the model's device for the flat parameter cotangents, or None
# (parallel.enable_peer_allreduce: the adjoint writes straight into the peer-mapped buffer the collective works on)
_flat_alloc = {}


def new_flat_grads(net, P, device):
    hook = _flat_alloc.get(id(net))
    if hook is not None:
        t = hook(P)
        if t is not None:
            return t
    return torch.empty(P, dtype=torch.float32, device=device)


def split_flat_grads(flat, G, H):
    """Views of the flat cotangent vector in the reference parameter order and shapes."""
    o, out = 0, []
    for shape in ((1, G), (H, G), (H,), (H, G), (H,), (G, 2 * H)):
        n = 1
        for d in shape:
            n *= d
        out.append(flat[o:o + n].view(shape))
        o += n
    return out


# ---- solves ----------------------------------------------------------------------------------------------------------------
def _zero_param_grads(net, G, H, device):
    """A single output time leaves nothing to integrate: the solution is y0 itself (solvers.py:26-30 fills solution[0]
    and the loop over the later times is empty) and the backward sweep (adjoint.py:137-154, an empty loop as well)
    returns grad_y[0] for y0 and ZERO -- not missing -- parameter cotangents."""
    flat = new_flat_grads(net, 4 * G * H + 2 * H + G, device)
    flat.zero_()
    return split_flat_grads(flat, G, H)


def _t_array(t_list):
    arr = (ctypes.c_double * len(t_list))(*t_list)
    return arr


# ---- fixed-grid step grids (options=dict(step_size=h); solvers.py:48-50, 77-103) -----------------------------------------
# Built here, once per call, with the reference's own tensor ops in the dtype of t (float32 or float64), so the steps and
# the interpolation slopes are the reference's bit for bit; the kernels only consume them (include/phoenix_b200.h, the
# *_grid entry points).
def fixed_grid(t, step_size):
    """The grid of ``FixedGridODESolver`` over the increasing 1-D tensor ``t`` (the solver's t, after the negation of a
    decreasing t), in t's dtype; raises the reference's AssertionError when it misses t[-1].  ``step_size``: a float or a
    0-dim CPU tensor, which takes part in the arithmetic with its own dtype, as in the reference."""
    niters = torch.ceil((t[-1] - t[0]) / step_size + 1).item()
    grid = torch.arange(0, niters, dtype=t.dtype) * step_size + t[0]
    if grid[-1] > t[-1]:
        grid[-1] = t[-1]
    assert grid[0] == t[0] and grid[-1] == t[-1]
    return grid


def forward_grid(t_list, t_is_f32, step_size):
    """One problem's forward grid: the float32 dt of every step, and for every output time t[j], j >= 1, the step whose
    end is the first grid point >= t[j] and the float32 slope (t[j] - t0) / (t1 - t0) of that step (-1: t[j] == t1)."""
    t = torch.tensor(t_list, dtype=torch.float32 if t_is_f32 else torch.float64)
    grid = fixed_grid(t, step_size)
    k = torch.searchsorted(grid[1:], t[1:])
    t0, t1 = grid[k], grid[k + 1]
    slope = torch.where(t[1:] == t1, -1.0, ((t[1:] - t0) / (t1 - t0)).float())
    return (grid[1:] - grid[:-1]).float(), k.to(torch.int32), slope.float()


def adjoint_grid(t_list, t_is_f32, step_size):
    """One problem's backward grids: the float32 dt of the steps of every interval [t[i], t[i+1]], each integrated on
    its own grid over the negated times [-t[i+1], -t[i]] (adjoint.py: odeint over t[i:i+2].flip(0)), and their counts."""
    dtype = torch.float32 if t_is_f32 else torch.float64
    dts = []
    for i in range(len(t_list) - 1):
        g = fixed_grid(torch.tensor([-t_list[i + 1], -t_list[i]], dtype=dtype), step_size)
        dts.append((g[1:] - g[:-1]).float())
    return torch.cat(dts), [int(d.numel()) for d in dts]


class _Grid:
    """Step grids of consecutive problems as phx_solve takes them (host arrays, kept alive here)."""

    def __init__(self, parts, forward):
        self.forward = forward
        self.dt = torch.cat([q[0] for q in parts]).contiguous()
        if forward:
            self.steps = torch.tensor([int(q[0].numel()) for q in parts], dtype=torch.int32)
            self.out_step = torch.cat([q[1] for q in parts]).contiguous()
            self.out_slope = torch.cat([q[2] for q in parts]).contiguous()
        else:
            self.steps = torch.tensor([n for q in parts for n in q[1]], dtype=torch.int32)

    def put(self, d):
        """Point the grid fields of the request ``d`` at these arrays."""
        d.grid_dt, d.grid_steps = self.dt.data_ptr(), self.steps.data_ptr()
        if self.forward:
            d.grid_out_step, d.grid_out_slope = self.out_step.data_ptr(), self.out_slope.data_ptr()

    def nbytes(self, lib, N, T):
        """Workspace room for the grid behind the solver's own part (16-byte alignment included)."""
        return 16 + lib.phx_grid_workspace_bytes(N, T, self.dt.numel())


def _grids(t_rows, t_is_f32, step_size, forward):
    """Per-problem grids (None without a step size: the calls stay the one-step-per-interval entry points)."""
    if step_size is None:
        return None
    build = forward_grid if forward else adjoint_grid
    return [build(r, t_is_f32, step_size) for r in t_rows]


_ENGINE_IDS = {"resident": _lib.ENGINE_RESIDENT, "rows": _lib.ENGINE_ROWS, "stream": _lib.ENGINE_STREAM}


def _solve_desc(engine, adjoint, packed, G, H, B, N, T, t_is_f32, method, rtol, atol, max_num_steps, param_mask=0,
                reversed_time=False, step_control=None, t_vjp=None):
    """The phx_solve request of a solve on ``engine`` ('resident' | 'rows' | 'stream'), with the fields all its launches
    share; each launch points it at its own times, state, workspace and status (_launch).  ``step_control``: dopri5's
    (first_step, safety, ifactor, dfactor), 0 for a default, or None for all four defaults.  ``t_vjp``: the adjoint's
    time cotangents [N, T-1] (time_vjp), or None for zero; a launch of a later problem points the request at its row."""
    d = _lib.PhxSolveDesc()
    d.engine, d.adjoint, d.G, d.H, d.B, d.N, d.T = _ENGINE_IDS[engine], int(adjoint), G, H, B, N, T
    d.packed, d.t_is_f32, d.reversed, d.method = packed.data_ptr(), int(t_is_f32), int(reversed_time), _lib.METHOD_IDS[method]
    d.rtol, d.atol, d.max_num_steps, d.param_mask = float(rtol), float(atol), int(max_num_steps), param_mask
    if step_control is not None:
        d.first_step, d.safety, d.ifactor, d.dfactor = (float(v) for v in step_control)
    if t_vjp is not None:
        d.t_vjp = t_vjp.data_ptr()
    return d


def _launch(lib, dev, d, t, ws, status, log, cap, what, stream=None):
    """phx_solve of ``d`` with the times ``t`` (a ctypes double array), workspace, status record(s) and step log given."""
    d.t_host = ctypes.addressof(t)
    d.workspace, d.workspace_bytes, d.status = ws.data_ptr(), ws.numel(), status.data_ptr()
    d.steplog, d.steplog_cap = (log.data_ptr(), cap) if log is not None else (None, 0)
    _lib.check(lib.phx_solve(_lib.ctx(dev), ctypes.byref(d), stream if stream is not None else _stream_ptr(dev)), what)


def _pick_engine(lib, dev, G, H, B, T, adjoint):
    """Resident (one persistent cooperative launch) when the rows fit on chip, else the streaming engine."""
    if FORCE_ENGINE != "stream" and B <= lib.phx_resident_max_rows(int(adjoint)):
        nb = lib.phx_solve_workspace_bytes(_lib.ctx(dev), G, H, B, T, int(adjoint))
        if nb > 0:
            return "resident", nb
    if FORCE_ENGINE == "resident":
        raise NotImplementedError("resident engine cannot take G=%d H=%d B=%d: %s" % (G, H, B, _lib.last_error()))
    nb = lib.phx_stream_workspace_bytes(_lib.ctx(dev), G, H, B, T, int(adjoint))
    if nb == 0:
        raise NotImplementedError("phoenix_b200: no kernel for G=%d H=%d B=%d (%s)" % (G, H, B, _lib.last_error()))
    return "stream", nb


_rows_cache = {}


def _rows_per_pass(lib, dev, G, H, adjoint):
    """Rows (independent one-row problems) the rows kernels advance per pass for this model; 0: not supported."""
    key = (dev, G, H, int(adjoint))
    r = _rows_cache.get(key)
    if r is None:
        r = _rows_cache[key] = int(lib.phx_rows_supported(_lib.ctx(dev), G, H, int(adjoint)))
    return r


def _use_rows(lib, dev, G, H, B, adjoint, single=False, T=2):
    """One-row problems go to the rows kernels (phx_rows.cuh) unless a test forces another engine -- or the call holds a
    single sample of a GPU-filling model and the one-problem resident kernels take it (SINGLE_CALL_ENGINE)."""
    if B != 1 or FORCE_ENGINE not in (None, "rows") or _rows_per_pass(lib, dev, G, H, adjoint) <= 0:
        return False
    if (single and FORCE_ENGINE is None and SINGLE_CALL_ENGINE == "resident" and G >= SINGLE_CALL_MIN_GENES
            and lib.phx_solve_workspace_bytes(_lib.ctx(dev), G, H, 1, T, int(adjoint)) > 0):
        return False
    return True


def _steplog_rows(n):
    tls = _tls()
    if not STEP_LOGGING:
        tls.last_log = None
        return None, 0
    log = torch.zeros(n, STEPLOG_CAP, 3, dtype=torch.float64).pin_memory()
    tls.last_log = log
    return log, STEPLOG_CAP


def _forward_rows(lib, net, packed, G, H, dev, y0c, t_rows, t_is_f32, reversed_time, method, rtol, atol, max_num_steps,
                  out_shape, grids=None, step_control=None):
    """N one-row problems (y0c [N, G]) in lock-step; returns yout of shape out_shape (= [N, T, ..., G] memory order).
    ``grids``: the problems' forward step grids (forward_grid), or None; ``step_control``: see _solve_desc."""
    N, T = len(t_rows), len(t_rows[0])
    nb = lib.phx_rows_workspace_bytes(_lib.ctx(dev), G, H, N, T, 0)
    grid = _Grid(grids, True) if grids is not None else None
    if grid is not None:
        nb += grid.nbytes(lib, N, T)
    ws = _workspace(dev, nb, "solve")
    yout = torch.empty(out_shape, dtype=torch.float32, device=y0c.device)
    stn = _new_status_block(N)
    log, cap = _steplog_rows(N)
    flat_t = (ctypes.c_double * (N * T))(*[x for r in t_rows for x in r])
    d = _solve_desc("rows", False, packed, G, H, 1, N, T, t_is_f32, method, rtol, atol, max_num_steps,
                    reversed_time=reversed_time, step_control=step_control)
    d.y0, d.y_out = y0c.data_ptr(), yout.data_ptr()
    if grid is not None:
        grid.put(d)
    _launch(lib, dev, d, flat_t, ws, stn, log, cap, "solve_forward_rows")
    _tls().last_status_block = stn
    for i in range(N):
        _finish(stn[i], "forward solve %d" % i if N > 1 else "forward solve", dev)
    return yout


def _adjoint_rows(lib, net, packed, G, H, dev, t_rows, t_is_f32, method, rtol, atol, max_num_steps, ys, gy, adj_shape,
                  param_mask=_lib.PARAMS_ALL, grids=None, step_control=None, t_vjp=None):
    """Backward sweeps of N one-row problems (ys, gy: [N, T, ..., G] memory order): adj_y0 and the SUM over the problems of
    the six parameter cotangents (flat, reference order; zeros for the parameters outside ``param_mask``).  ``grids``:
    the problems' backward step grids (adjoint_grid), or None; ``step_control``, ``t_vjp`` ([N, T-1]): see _solve_desc."""
    N, T = len(t_rows), len(t_rows[0])
    nb = lib.phx_rows_workspace_bytes(_lib.ctx(dev), G, H, N, T, 1)
    grid = _Grid(grids, False) if grids is not None else None
    if grid is not None:
        nb += grid.nbytes(lib, N, T)
    ws = _workspace(dev, nb, "solve")
    adj_y0 = torch.empty(adj_shape, dtype=torch.float32, device=ys.device)
    ctx = _lib.ctx(dev)
    parts = lib.phx_rows_grad_parts(ctx, G, H, N)
    gpk = _workspace(dev, parts * lib.phx_packed_grad_bytes(G, H), "gradparts")
    P = 4 * G * H + 2 * H + G
    flat = new_flat_grads(net, P, ys.device)
    stn = _new_status_block(N)
    log, cap = _steplog_rows(N)
    flat_t = (ctypes.c_double * (N * T))(*[x for r in t_rows for x in r])
    sp = _stream_ptr(dev)
    d = _solve_desc("rows", True, packed, G, H, 1, N, T, t_is_f32, method, rtol, atol, max_num_steps, param_mask,
                    step_control=step_control, t_vjp=t_vjp)
    d.y_saved, d.grad_y, d.adj_y0, d.grads = ys.data_ptr(), gy.data_ptr(), adj_y0.data_ptr(), gpk.data_ptr()
    if grid is not None:
        grid.put(d)
    _launch(lib, dev, d, flat_t, ws, stn, log, cap, "solve_adjoint_rows", sp)
    _lib.check(lib.phx_unpack_grads_masked(ctx, G, H, _ptr(gpk), parts, _ptr(flat), 0, param_mask & _lib.PARAMS_ALL,
                                           sp), "unpack_grads")
    _tls().last_status_block = stn
    for i in range(N):
        _finish(stn[i], "adjoint solve %d" % i if N > 1 else "adjoint solve", dev)
    return adj_y0, split_flat_grads(flat, G, H)


@_on_model_device
def solve_forward(net, y0, t_list, t_is_f32, reversed_time, method, rtol, atol, max_num_steps, step_size=None,
                  step_control=None):
    """``step_size`` (fixed-grid methods): integrate on the reference's grid of that spacing and interpolate the output
    times inside a step (solvers.py:48-50, 77-103); None: one step per output interval.  ``step_control`` (dopri5):
    (first_step, safety, ifactor, dfactor), 0 for a default (include/phoenix_b200.h, phx_solve), or None."""
    packed, G, H, dev = packed_weights(net)
    if y0.shape[-1] != G:
        raise RuntimeError("last dimension of y0 (%d) must equal ndim (%d)" % (y0.shape[-1], G))
    if _device_index(y0) != dev:
        raise RuntimeError("y0 and the ODENet parameters must be on the same CUDA device")
    y0c = y0.detach().contiguous()
    B = y0c.numel() // G
    T = len(t_list)
    if T == 1:
        return y0c.unsqueeze(0).clone()
    lib = _lib.load()
    grids = _grids([t_list], t_is_f32, step_size, True)
    if _use_rows(lib, dev, G, H, B, False, single=True, T=T):
        return _forward_rows(lib, net, packed, G, H, dev, y0c, [t_list], t_is_f32, reversed_time, method, rtol, atol,
                             max_num_steps, (T,) + tuple(y0c.shape), grids, step_control)
    engine, nb = _pick_engine(lib, dev, G, H, B, T, False)
    grid = _Grid(grids, True) if grids is not None else None
    if grid is not None and engine == "resident":
        nb += grid.nbytes(lib, 1, T)
    ws = _workspace(dev, nb, "solve" if engine == "resident" else "stream")
    yout = torch.empty((T,) + tuple(y0c.shape), dtype=torch.float32, device=y0c.device)
    st = _new_status()
    log, cap = _steplog()
    d = _solve_desc(engine, False, packed, G, H, B, 1, T, t_is_f32, method, rtol, atol, max_num_steps,
                    reversed_time=reversed_time, step_control=step_control)
    d.y0, d.y_out = y0c.data_ptr(), yout.data_ptr()
    if grid is not None:
        grid.put(d)
    _launch(lib, dev, d, _t_array(t_list), ws, st, log, cap, "solve_forward")
    _finish(st, "forward solve", dev)
    return yout


@_on_model_device
def solve_adjoint(net, t_list, t_is_f32, method, rtol, atol, max_num_steps, y_saved, grad_y,
                  param_mask=_lib.PARAMS_ALL, step_size=None, step_control=None, t_vjp=None):
    """adj_y0 and the six parameter cotangents of one backward sweep.  ``param_mask`` (bit i = the i-th parameter in
    reference order): the adjoint parameters, the only ones integrated and put in the error norm; the cotangents of the
    others come back as zeros.  With ``_lib.NORM_SEMINORM`` also set, the dopri5 error norm leaves the parameter block
    out altogether (the seminorm).  ``step_size`` (fixed-grid methods): every interval is integrated on its own grid of
    that spacing (adjoint_grid); None: one step per interval.  ``step_control``: as in solve_forward, with first_step the
    first dt of every interval.  ``t_vjp``: the time cotangent entering each interval, [1, T-1] float32 on the device
    (time_vjp), when t needs a gradient; None: zero."""
    packed, G, H, dev = packed_weights(net)
    ys = y_saved.detach().contiguous()
    gy = grad_y.detach().to(torch.float32).contiguous()
    T = len(t_list)
    if T == 1:
        return gy[0].clone(), _zero_param_grads(net, G, H, ys.device)
    B = ys[0].numel() // G
    lib = _lib.load()
    grids = _grids([t_list], t_is_f32, step_size, False)
    if _use_rows(lib, dev, G, H, B, True, single=True, T=T):
        return _adjoint_rows(lib, net, packed, G, H, dev, [t_list], t_is_f32, method, rtol, atol, max_num_steps, ys, gy,
                             tuple(ys[0].shape), param_mask, grids, step_control, t_vjp)
    engine, nb = _pick_engine(lib, dev, G, H, B, T, True)
    grid = _Grid(grids, False) if grids is not None else None
    if grid is not None and engine == "resident":
        nb += grid.nbytes(lib, 1, T)
    ws = _workspace(dev, nb, "solve" if engine == "resident" else "stream")
    adj_y0 = torch.empty_like(ys[0])
    P = 4 * G * H + 2 * H + G
    grads = new_flat_grads(net, P, ys.device)
    st = _new_status()
    log, cap = _steplog()
    d = _solve_desc(engine, True, packed, G, H, B, 1, T, t_is_f32, method, rtol, atol, max_num_steps, param_mask,
                    step_control=step_control, t_vjp=t_vjp)
    d.y_saved, d.grad_y, d.adj_y0, d.grads = ys.data_ptr(), gy.data_ptr(), adj_y0.data_ptr(), grads.data_ptr()
    if grid is not None:
        grid.put(d)
    _launch(lib, dev, d, _t_array(t_list), ws, st, log, cap, "solve_adjoint")
    _finish(st, "adjoint solve", dev)
    return adj_y0, split_flat_grads(grads, G, H)


@_on_model_device
def time_vjp(net, y_saved, grad_y):
    """The time cotangents of N adjoint backwards (adjoint.py, backward with t requiring grad) from the saved outputs and
    their cotangents ``[N, T, *S, G]``: ``(t_grad [N, T], t_vjp [N, T-1])``, float32 on the device.  t_grad is the
    gradient with respect to each problem's t; t_vjp[:, i] is the time cotangent the reference carries through the
    interval [t[i], t[i+1]], what solve_adjoint / solve_adjoint_many take to start dopri5 there as the reference does.
    No sweep is needed for them: the RHS is autonomous (include/phoenix_b200.h, phx_time_vjp)."""
    packed, G, H, dev = packed_weights(net)
    ys = y_saved.detach().contiguous()
    gy = grad_y.detach().to(torch.float32).contiguous()
    N, T = ys.shape[0], ys.shape[1]
    B = ys[0, 0].numel() // G
    t_grad = torch.empty(N, T, dtype=torch.float32, device=ys.device)
    t_vjp = torch.empty(N, T - 1, dtype=torch.float32, device=ys.device)
    lib = _lib.load()
    nb = lib.phx_time_vjp_workspace_bytes(G, H, B, N, T)
    ws = _workspace(dev, nb, "tvjp")   # (not the "rhs" one: that may still hold [S|P] for a pending rhs_vjp)
    _lib.check(lib.phx_time_vjp(_lib.ctx(dev), G, H, B, N, T, _ptr(packed), _ptr(ys), _ptr(gy), _ptr(t_grad),
                                _ptr(t_vjp), _ptr(ws), ws.numel(), _stream_ptr(dev)), "time_vjp")
    return t_grad, t_vjp


# ---- many independent problems per call (SURVEY.md section 8 f1: the per-sample loop of training_step) -----------------
_MANY_CHUNK = 32   # samples whose [P]-long parameter cotangents are held at once before they are summed


def _t_rows(t_rows):
    return [(ctypes.c_double * len(r))(*r) for r in t_rows]


def _problems_per_launch(T):
    return max(1, 16 // T)   # PHX_T_INLINE output times travel with the kernel parameters


def _new_status_block(n):
    """n contiguous pinned status records (one per problem of a multi-problem launch), all marked RUNNING."""
    _poll_pending()
    words = ctypes.sizeof(_lib.PhxStatus) // 4
    st = torch.empty(n, words, dtype=torch.int32).pin_memory()
    ctypes.memset(st.data_ptr(), 0, n * ctypes.sizeof(_lib.PhxStatus))
    for i in range(n):
        _lib.PhxStatus.from_address(st.data_ptr() + i * ctypes.sizeof(_lib.PhxStatus)).code = _lib.ST_RUNNING
    return st


_MANY_MAX_STREAMS = 8
_side_streams = {}


def _concurrency(lib, dev, G, H, B, adjoint, engine, n_problems):
    """How many of the independent solves can run side by side: a resident solve of a small model occupies only
    ceil(G / 16) of the SMs (22 CTAs at 350 genes, 44 at 690), so several persistent launches fit on the GPU at once --
    each on its own stream with its own workspace.  Genome-scale models fill the GPU by themselves (1)."""
    if engine != "resident" or n_problems < 2:
        return []
    out = (ctypes.c_int32 * 8)()
    num_sms = lib.phx_ctx_num_sms(_lib.ctx(dev))
    if lib.phx_plan_describe(num_sms, G, H, B, int(adjoint), out) != _lib.PHX_OK:
        return []
    k = min(num_sms // max(1, out[0]), _MANY_MAX_STREAMS, n_problems)
    if k < 2:
        return []
    pool = _side_streams.setdefault(dev, [])
    while len(pool) < k:
        pool.append(torch.cuda.Stream(device=dev))
    return pool[:k]


def _fan_out(dev, streams):
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream(dev))
    for st in streams:
        st.wait_event(ev)


def _fan_in(dev, streams):
    main = torch.cuda.current_stream(dev)
    for st in streams:
        ev = torch.cuda.Event()
        ev.record(st)
        main.wait_event(ev)


@_on_model_device
def solve_forward_many(net, y0, t_rows, t_is_f32, method, rtol, atol, max_num_steps, step_size=None, step_control=None):
    """y0 ``[N, *S, G]``: N independent problems, problem i integrated over its own times ``t_rows[i]`` (all of length
    T).  Every problem is one resident launch with its own step controller -- exactly the reference's per-sample call
    (train_insilico.py:128-130) -- but the weights are packed, the workspace fetched and the arguments marshalled once
    for the whole set.  Returns ``[N, T, *S, G]``.  ``step_size``: as in solve_forward, every problem on its own grid;
    ``step_control``: as in solve_forward."""
    packed, G, H, dev = packed_weights(net)
    if y0.shape[-1] != G:
        raise RuntimeError("last dimension of y0 (%d) must equal ndim (%d)" % (y0.shape[-1], G))
    if _device_index(y0) != dev:
        raise RuntimeError("y0 and the ODENet parameters must be on the same CUDA device")
    y0c = y0.detach().contiguous()
    N, T = len(t_rows), len(t_rows[0])
    if T == 1:
        return y0c.unsqueeze(1).clone()
    B = y0c[0].numel() // G
    lib = _lib.load()
    grids = _grids(t_rows, t_is_f32, step_size, True)
    if _use_rows(lib, dev, G, H, B, False):
        return _forward_rows(lib, net, packed, G, H, dev, y0c, t_rows, t_is_f32, False, method, rtol, atol, max_num_steps,
                             (N, T) + tuple(y0c.shape[1:]), grids, step_control)
    engine, nb = _pick_engine(lib, dev, G, H, B, T, False)
    if grids is not None and engine == "resident":
        nb += _Grid(grids, True).nbytes(lib, N, T)
    ws = _workspace(dev, nb, "solve" if engine == "resident" else "stream")
    yout = torch.empty((N, T) + tuple(y0c.shape[1:]), dtype=torch.float32, device=y0c.device)
    sp = _stream_ptr(dev)
    ybase, obase = y0c.data_ptr(), yout.data_ptr()
    ystride, ostride = y0c[0].numel() * 4, yout[0].numel() * 4
    tarr = _t_rows(t_rows)
    streams = _concurrency(lib, dev, G, H, B, False, engine, N)
    if streams:
        _fan_out(dev, streams)
    per = _problems_per_launch(T) if (engine == "resident" and not streams and not STEP_LOGGING) else 1
    d = _solve_desc(engine, False, packed, G, H, B, 1, T, t_is_f32, method, rtol, atol, max_num_steps,
                    step_control=step_control)
    if per > 1:
        # genome-scale model: a solve fills the GPU, so the problems go through ONE persistent launch a few at a time
        # and the weights are staged on chip once per launch instead of once per problem
        for lo in range(0, N, per):
            n = min(per, N - lo)
            stn = _new_status_block(n)
            flat_t = (ctypes.c_double * (n * T))(*[x for r in t_rows[lo:lo + n] for x in r])
            d.N, d.y0, d.y_out = n, ybase + lo * ystride, obase + lo * ostride
            if grids is not None:
                gm = _Grid(grids[lo:lo + n], True)
                gm.put(d)
            _launch(lib, dev, d, flat_t, ws, stn, None, 0, "solve_forward_many", sp)
            for i in range(n):
                _finish(stn[i], "forward solve %d" % (lo + i), dev)
        return yout
    pg = [_Grid([g], True) for g in grids] if grids is not None else None   # (kept alive over the calls)
    try:   # an error raised for one problem must not leave the caller's stream un-ordered after the side streams
        for i in range(N):
            st = _new_status()
            log, cap = _steplog()
            d.y0, d.y_out = ybase + i * ystride, obase + i * ostride
            if pg is not None:
                pg[i].put(d)
            if streams:
                with torch.cuda.stream(streams[i % len(streams)]):
                    _launch(lib, dev, d, tarr[i], _workspace(dev, nb, "solve"), st, log, cap, "solve_forward")
                    _finish(st, "forward solve %d" % i, dev)
                continue
            _launch(lib, dev, d, tarr[i], ws, st, log, cap, "solve_forward", sp)
            _finish(st, "forward solve %d" % i, dev)
    finally:
        if streams:
            _fan_in(dev, streams)
    return yout


@_on_model_device
def solve_adjoint_many(net, t_rows, t_is_f32, method, rtol, atol, max_num_steps, y_saved, grad_y,
                       param_mask=_lib.PARAMS_ALL, step_size=None, step_control=None, t_vjp=None):
    """Backward sweeps of N independent problems (``y_saved``, ``grad_y``: ``[N, T, *S, G]``): adj_y0 ``[N, *S, G]`` and
    the six parameter cotangents summed over the problems (what autograd accumulates into ``.grad``); zeros for the
    parameters outside ``param_mask``; ``step_size``, ``step_control``: see solve_adjoint; ``t_vjp``: [N, T-1], row i
    for problem i, see solve_adjoint)."""
    packed, G, H, dev = packed_weights(net)
    ys = y_saved.detach().contiguous()
    gy = grad_y.detach().to(torch.float32).contiguous()
    N, T = len(t_rows), len(t_rows[0])
    if T == 1:
        return gy[:, 0].clone(), _zero_param_grads(net, G, H, ys.device)
    B = ys[0, 0].numel() // G
    lib = _lib.load()
    grids = _grids(t_rows, t_is_f32, step_size, False)
    if _use_rows(lib, dev, G, H, B, True):
        return _adjoint_rows(lib, net, packed, G, H, dev, t_rows, t_is_f32, method, rtol, atol, max_num_steps, ys, gy,
                             tuple(ys[:, 0].shape), param_mask, grids, step_control, t_vjp)
    engine, nb = _pick_engine(lib, dev, G, H, B, T, True)
    if grids is not None and engine == "resident":
        nb += _Grid(grids, False).nbytes(lib, N, T)
    ws = _workspace(dev, nb, "solve" if engine == "resident" else "stream")
    adj_y0 = torch.empty_like(ys[:, 0])
    P = 4 * G * H + 2 * H + G
    chunk = min(N, _MANY_CHUNK)
    grads = torch.empty(chunk, P, dtype=torch.float32, device=ys.device)
    total = None
    pg = [_Grid([g], False) for g in grids] if grids is not None else None   # (kept alive over the calls)
    sp = _stream_ptr(dev)
    ybase, gbase, abase, tbase = ys.data_ptr(), gy.data_ptr(), adj_y0.data_ptr(), grads.data_ptr()
    stride = ys[0].numel() * 4
    astride = adj_y0[0].numel() * 4
    tarr = _t_rows(t_rows)
    streams = _concurrency(lib, dev, G, H, B, True, engine, N)
    per = _problems_per_launch(T) if (engine == "resident" and not streams and not STEP_LOGGING) else 1
    d = _solve_desc(engine, True, packed, G, H, B, 1, T, t_is_f32, method, rtol, atol, max_num_steps, param_mask,
                    step_control=step_control, t_vjp=t_vjp)
    tv_row = 4 * (T - 1)   # bytes between the t_vjp rows of consecutive problems
    for lo in range(0, N, chunk):
        hi = min(N, lo + chunk)
        if per > 1:
            for l2 in range(lo, hi, per):
                n = min(per, hi - l2)
                stn = _new_status_block(n)
                flat_t = (ctypes.c_double * (n * T))(*[x for r in t_rows[l2:l2 + n] for x in r])
                d.N, d.y_saved, d.grad_y = n, ybase + l2 * stride, gbase + l2 * stride
                d.adj_y0, d.grads = abase + l2 * astride, tbase + (l2 - lo) * P * 4
                if t_vjp is not None:
                    d.t_vjp = t_vjp.data_ptr() + l2 * tv_row
                if grids is not None:
                    gm = _Grid(grids[l2:l2 + n], False)
                    gm.put(d)
                _launch(lib, dev, d, flat_t, ws, stn, None, 0, "solve_adjoint_many", sp)
                for i in range(n):
                    _finish(stn[i], "adjoint solve %d" % (l2 + i), dev)
            part = grads[:hi - lo].sum(dim=0)
            total = part if total is None else total + part
            continue
        if streams:
            _fan_out(dev, streams)
        try:
            for i in range(lo, hi):
                st = _new_status()
                log, cap = _steplog()
                d.y_saved, d.grad_y = ybase + i * stride, gbase + i * stride
                d.adj_y0, d.grads = abase + i * astride, tbase + (i - lo) * P * 4
                if t_vjp is not None:
                    d.t_vjp = t_vjp.data_ptr() + i * tv_row
                if pg is not None:
                    pg[i].put(d)
                if streams:
                    with torch.cuda.stream(streams[i % len(streams)]):
                        _launch(lib, dev, d, tarr[i], _workspace(dev, nb, "solve"), st, log, cap, "solve_adjoint")
                        _finish(st, "adjoint solve %d" % i, dev)
                    continue
                _launch(lib, dev, d, tarr[i], ws, st, log, cap, "solve_adjoint", sp)
                _finish(st, "adjoint solve %d" % i, dev)
        finally:
            if streams:
                _fan_in(dev, streams)
        part = grads[:hi - lo].sum(dim=0)
        total = part if total is None else total + part
    return adj_y0, split_flat_grads(total, G, H)
