"""``odeint`` / ``odeint_adjoint`` with the reference's call surface (torchdiffeq/_impl/odeint.py:25-69,
adjoint.py:165-204) — argument normalisation follows misc.py:165-241 — dispatching to the CUDA solvers."""
import threading
import warnings
import weakref

import torch
import torch.nn as nn

from .. import engine
from .._lib import NORM_SEMINORM, PARAMS_ALL
from ..odenet import ODENet

# every method string the vendored package registers (odeint.py:9-22); only the four PHOENIX uses are accelerated
_REFERENCE_SOLVERS = ('dopri8', 'dopri5', 'bosh3', 'adaptive_heun', 'euler', 'midpoint', 'rk4', 'explicit_adams',
                      'implicit_adams', 'fixed_adams')
_SUPPORTED = ('dopri5', 'euler', 'midpoint', 'rk4')
_DEFAULT_MAX_STEPS = 2 ** 31 - 1


_FIXED_GRID = ('euler', 'midpoint', 'rk4')


def _step_size(method, options):
    """The fixed-grid ``step_size`` option (solvers.py:48-50), or None when it is not given: a float, or for a tensor
    ``(value, dtype)``.  A tensor keeps its dtype because the reference builds the grid under tensor type promotion (a
    0-dim float64 step size makes the step count of a float32 t's grid a float64 division); the pair keeps the deferred
    adjoint's group key hashable (_stepped turns it back into the tensor).  Only the three fixed-grid methods take it
    (dopri5: the generic refusal of _normalise); ``grid_constructor`` is refused."""
    if not options:
        return None
    if 'grid_constructor' in options:
        raise NotImplementedError("options['grid_constructor'] is not supported on the B200 path: the backward would call "
                                  "it with the augmented dynamics and state, which exist only on the device; use "
                                  "step_size")
    if 'step_size' not in options or (method or 'dopri5') not in _FIXED_GRID:
        return None
    h = options['step_size']
    if torch.is_tensor(h) and h.dim() != 0:
        raise NotImplementedError("a tensor step_size must be 0-dimensional (got shape {})".format(tuple(h.shape)))
    v = float(h.item() if torch.is_tensor(h) else h)
    if not (v > 0 and v != float('inf')):
        raise ValueError("step_size must be a positive finite number (got {})".format(options['step_size']))
    return (v, h.dtype) if torch.is_tensor(h) else v


_STEP_CONTROL = ('first_step', 'safety', 'ifactor', 'dfactor')


def _step_control(method, options):
    """The dopri5 step-control options (rk_common.py:111-228, misc.py:94-103) as a tuple of floats (first_step, safety,
    ifactor, dfactor), 0.0 for one not given (the engine's default: Hairer's initial-step estimate, 0.9, 10, 0.2), or
    None when none of them is given.  Only dopri5 takes them (the fixed-grid methods: the generic refusal of
    _normalise).  Non-positive or non-finite values are refused: the reference would loop or hit its underflow
    assertion."""
    if not options or (method or 'dopri5') != 'dopri5' or not any(k in options for k in _STEP_CONTROL):
        return None
    out = []
    for k in _STEP_CONTROL:
        if k not in options:
            out.append(0.0)
            continue
        v = options[k]
        if torch.is_tensor(v) and v.dim() != 0:
            raise NotImplementedError("a tensor {} must be 0-dimensional (got shape {})".format(k, tuple(v.shape)))
        f = float(v)
        if not (f > 0 and f != float('inf')):
            raise ValueError("{} must be a positive finite number (got {})".format(k, v))
        out.append(f)
    return tuple(out)


def _normalise(func, y0, t, rtol, atol, method, options):
    """The checks of misc.py:165-241 that apply to a single-tensor state; returns the pieces the kernels need (the
    fixed-grid ``step_size`` and the dopri5 step control are checked here and read with _step_size / _step_control)."""
    if not torch.is_tensor(y0):
        assert isinstance(y0, tuple), 'y0 must be either a torch.Tensor or a tuple'
        raise NotImplementedError("tuple-valued states are not part of the PHOENIX path (ODENet has a tensor state)")
    if not torch.is_floating_point(y0):
        raise TypeError('`y0` must be a floating point Tensor but is a {}'.format(y0.type()))
    options = {} if options is None else dict(options)
    if method is None:
        method = 'dopri5'
    if method not in _REFERENCE_SOLVERS:
        raise ValueError('Invalid method "{}". Must be one of {}'.format(
            method, '{"' + '", "'.join(_REFERENCE_SOLVERS) + '"}.'))
    if method not in _SUPPORTED:
        raise NotImplementedError('method "{}" is registered by torchdiffeq but never selected by PHOENIX; the B200 '
                                  'path implements {}'.format(method, _SUPPORTED))
    max_num_steps = int(options.pop('max_num_steps', _DEFAULT_MAX_STEPS))
    options.pop('dtype', None)
    if _step_size(method, options) is not None:
        options.pop('step_size')
    if _step_control(method, options) is not None:
        for k in _STEP_CONTROL:
            options.pop(k, None)
    if options:
        raise NotImplementedError("solver options {} are not supported on the B200 path with method {!r} (it takes "
                                  "max_num_steps and dtype; dopri5 also first_step, safety, ifactor and dfactor; "
                                  "euler, midpoint and rk4 also step_size)".format(sorted(options), method))
    assert torch.is_tensor(t), 't must be a torch.Tensor'
    assert t.ndimension() == 1, "{} must be one dimensional".format('t')
    if not torch.is_floating_point(t):
        raise TypeError('`{}` must be a floating point Tensor but is a {}'.format('t', t.type()))
    if t.requires_grad:
        raise NotImplementedError("gradients with respect to t are not computed on the B200 path")
    # the times are consumed on the host (float32 values are promoted exactly, like solvers.py:26); plain Python from
    # here on: this runs once per sample of every training step
    t_is_f32 = t.dtype != torch.float64
    tl = t.tolist()
    reversed_time = False
    if len(tl) > 1 and all(b < a for a, b in zip(tl, tl[1:])):
        tl = [-x for x in tl]
        reversed_time = True
    assert all(b > a for a, b in zip(tl, tl[1:])), '{} must be strictly increasing or decreasing'.format('t')
    if torch.is_tensor(rtol):
        assert not rtol.requires_grad, "rtol cannot require gradient"
        rtol = float(rtol)
    if torch.is_tensor(atol):
        assert not atol.requires_grad, "atol cannot require gradient"
        atol = float(atol)
    if not isinstance(func, ODENet):
        raise TypeError("phoenix_b200.torchdiffeq integrates phoenix ODENet right-hand sides only (got {}); there is "
                        "no generic / CPU fallback".format(type(func).__name__))
    if y0.dtype != torch.float32:
        raise TypeError("the B200 path keeps the state in float32 like the reference (got {})".format(y0.dtype))
    return tl, t_is_f32, reversed_time, float(rtol), float(atol), method, max_num_steps


def odeint(func, y0, t, rtol=1e-7, atol=1e-9, method=None, options=None):
    """Integrate dy/dt = func(t, y) from y(t[0]) = y0 and return y at every t: ``[len(t), *y0.shape]``
    (odeint.py:25-69).  Not differentiable — use ``odeint_adjoint`` (what every PHOENIX script imports as ``odeint``,
    train_insilico.py:15-18) when gradients are needed."""
    tl, t_is_f32, rev, rtol, atol, method, max_steps = _normalise(func, y0, t, rtol, atol, method, options)
    step, ctl = _step_size(method, options), _step_control(method, options)
    if torch.is_grad_enabled() and (y0.requires_grad or any(p.requires_grad for p in func.parameters())):
        warnings.warn("phoenix_b200.odeint does not record an autograd graph; use odeint_adjoint for gradients",
                      stacklevel=2)
    with torch.no_grad():
        return engine.solve_forward(func, y0, tl, t_is_f32, rev, method, rtol, atol, max_steps, **_stepped(step),
                                    **_controlled((ctl,), 0))


# ---- the per-sample loop of training_step, backward side ----------------------------------------------------------------
# train_insilico.py:128-130 calls odeint once per sample and backpropagates one loss, so autograd meets N independent
# adjoint nodes of the same model in one backward pass.  Each is a one-row problem, and a pass of the rows kernels
# costs the same with one row as with four (DESIGN 3.1b) -- so the nodes of one backward pass hand their cotangents to
# the LAST of them to run, which solves all the sweeps in one lock-step call (engine.solve_adjoint_many, the backward of
# odeint_adjoint_many) and returns the summed parameter cotangents as its own; the others return None (= zero).  What
# autograd accumulates -- into .grad or into torch.autograd.grad's outputs -- is the same sum.  A node whose y0 needs a
# gradient, or that is alone in its pass, runs its own sweep as before.
DEFER_ADJOINT = True
_NOT_DEFERRED = object()
_defer_lock = threading.RLock()
_live_nodes = weakref.WeakKeyDictionary()   # ODENet -> WeakSet of adjoint nodes (autograd contexts) built on it
_deferred = {}                               # (graph task id, group key) -> [expected count, [(seq, y, grad_y, tl), ...]]
_node_seq = [0]


def set_deferred_adjoint(flag):
    """Batch the backward sweeps of the per-sample ``odeint_adjoint`` nodes of one backward pass (default on)."""
    global DEFER_ADJOINT
    DEFER_ADJOINT = bool(flag)


def _register_node(ctx, func, y0, tl, t_is_f32, adj):
    """Forward side: note the node if its backward may be batched with its siblings' (a one-row state that needs no
    gradient itself -- the training loop's case)."""
    ctx.group = None
    if (not DEFER_ADJOINT or ctx.needs_input_grad[8] or not any(ctx.needs_input_grad[9:]) or not adj[4] & PARAMS_ALL
            or y0.numel() != y0.shape[-1]):
        return   # (nothing to differentiate -- e.g. a validation pass under no_grad -- is not a node at all)
    with _defer_lock:
        _node_seq[0] += 1
        ctx.seq = _node_seq[0]
        # adj[4], the adjoint parameter mask with the norm bit, adj[5], the backward step size, and adj[6], its dopri5
        # step control when given, are part of the key: only nodes with the same adjoint set, error norm, step grid spacing and
        # controller share a sweep
        ctx.group = (len(tl), t_is_f32, adj, tuple(y0.shape), y0.device, tuple(ctx.needs_input_grad[9:]))
        nodes = _live_nodes.get(func)
        if nodes is None:
            nodes = _live_nodes[func] = weakref.WeakSet()
        nodes.add(ctx)


def _unresolved(key):
    def check():
        with _defer_lock:
            ent = _deferred.pop(key, None)
        if ent is not None:
            raise RuntimeError("phoenix_b200: %d of %d odeint_adjoint nodes of this backward pass handed their cotangents "
                               "to a sibling that never ran, so their parameter gradients are missing; call "
                               "phoenix_b200.torchdiffeq.set_deferred_adjoint(False) and report this"
                               % (len(ent[1]), ent[0]))
    return check


def _defer(ctx, y, grad_y):
    """Backward side.  Returns _NOT_DEFERRED (the caller solves its own sweep), the all-None tuple (the cotangent waits for
    the last sibling) or, in the last sibling, (t_rows, ys, gys) of every waiting node in creation order."""
    try:
        gid = torch._C._current_graph_task_id()
        will_run = torch._C._will_engine_execute_node
        queue_callback = torch.autograd.Variable._execution_engine.queue_callback
    except AttributeError:
        return _NOT_DEFERRED
    if gid < 0:
        return _NOT_DEFERRED
    key = (gid, id(ctx.func), ctx.group)
    with _defer_lock:
        ent = _deferred.get(key)
        if ent is None:
            try:
                peers = [c for c in list(_live_nodes.get(ctx.func, ())) if c.group == ctx.group and will_run(c)]
            except Exception:
                return _NOT_DEFERRED
            if len(peers) < 2 or not any(c is ctx for c in peers):
                return _NOT_DEFERRED
            for k in [k for k in _deferred if k[0] < gid - 8]:   # passes that died with an exception
                del _deferred[k]
            ent = _deferred[key] = [len(peers), []]
            queue_callback(_unresolved(key))   # runs when this backward pass ends: loud if a counted sibling never came
        ent[1].append((ctx.seq, y, grad_y, ctx.tl))
        if len(ent[1]) < ent[0]:
            return None
        del _deferred[key]
    items = sorted(ent[1], key=lambda it: it[0])
    return [it[3] for it in items], torch.stack([it[1] for it in items]), torch.stack([it[2] for it in items])


class OdeintAdjointMethod(torch.autograd.Function):
    """adjoint.py:10-162: forward = solve under no_grad, keep only y(t); backward = one device-side sweep of the
    augmented system per output interval (batched with the sibling nodes of the same backward pass, see above)."""

    @staticmethod
    def forward(ctx, func, tl, t_is_f32, fwd, rtol, atol, max_steps, adj, y0, *adjoint_params):
        # fwd = (method, step_size); adj = (method, rtol, atol, max_num_steps, mask, step_size) of the backward; each
        # with the dopri5 step control appended when it is given (_with_control)
        ctx.func, ctx.tl, ctx.t_is_f32, ctx.adj = func, tl, t_is_f32, adj
        with torch.no_grad():
            y = engine.solve_forward(func, y0, tl, t_is_f32, False, fwd[0], rtol, atol, max_steps, **_stepped(fwd[1]),
                                     **_controlled(fwd, 2))
        ctx.save_for_backward(y)
        _register_node(ctx, func, y0, tl, t_is_f32, adj)
        return y

    @staticmethod
    def backward(ctx, grad_y):
        (y,) = ctx.saved_tensors
        a_method, a_rtol, a_atol, a_max, mask = ctx.adj[:5]
        if not mask & PARAMS_ALL and not ctx.needs_input_grad[8]:
            return (None,) * (9 + len(ctx.needs_input_grad[9:]))   # only parameters outside adjoint_params want one
        batch = _defer(ctx, y, grad_y) if (ctx.group is not None and DEFER_ADJOINT) else _NOT_DEFERRED
        if batch is None:
            return (None,) * (9 + len(ctx.needs_input_grad[9:]))
        kw = dict(_masked(mask), **_stepped(ctx.adj[5]), **_controlled(ctx.adj, 6))
        with torch.no_grad():
            if batch is _NOT_DEFERRED:
                adj_y0, grads = engine.solve_adjoint(ctx.func, ctx.tl, ctx.t_is_f32, a_method, a_rtol, a_atol, a_max,
                                                     y, grad_y, **kw)
            else:
                t_rows, ys, gys = batch
                adj_y0, grads = engine.solve_adjoint_many(ctx.func, t_rows, ctx.t_is_f32, a_method, a_rtol, a_atol,
                                                          a_max, ys, gys, **kw)
        return _grads_out(ctx, adj_y0, grads, mask)


def _masked(mask):
    """The engine's keyword for a proper subset of the parameters or the seminorm; with all six parameters and the
    default norm the engine is called as it always was."""
    return {} if mask == PARAMS_ALL else {"param_mask": mask}


def _stepped(step_size):
    """The engine's keyword for a fixed-grid step size (_step_size's form: a float, or (value, dtype) of a tensor);
    without one the engine is called as it always was."""
    if step_size is None:
        return {}
    if isinstance(step_size, tuple):
        return {"step_size": torch.tensor(step_size[0], dtype=step_size[1])}
    return {"step_size": step_size}


def _with_control(tup, step_control):
    """The fwd / adj tuple of an adjoint node with the dopri5 step control (_step_control's tuple) appended; without one
    the tuple is what it always was."""
    return tup if step_control is None else tup + (step_control,)


def _controlled(tup, i):
    """The engine's keyword for the step control at tup[i] (_with_control); without one the engine is called as it always
    was."""
    return {} if len(tup) <= i or tup[i] is None else {"step_control": tup[i]}


def _grads_out(ctx, adj_y0, grads, mask):
    """backward's result: adj_y0 for y0, and a cotangent only for the parameters in the adjoint set (None for the others
    even when they require grad: the reference's adjoint node does not take them as inputs).  Only the six parameter bits
    of ``mask`` are read, never the norm bit."""
    out = [None] * 8 + [adj_y0 if ctx.needs_input_grad[8] else None]
    for i, need in enumerate(ctx.needs_input_grad[9:]):
        out.append(grads[i] if (need and mask >> i & 1) else None)
    return tuple(out)


def _adjoint_mask(func, adjoint_params):
    """The six ODENet parameters and the mask (bit i = the i-th in reference order) of the adjoint set S: the members of
    ``adjoint_params`` -- all six when None -- that require grad (adjoint.py:185-193)."""
    params = engine.net_params(func)
    if adjoint_params is None:
        chosen = params
    else:
        chosen = list(adjoint_params)
        ids = [id(p) for p in params]
        seen = set()
        for p in chosen:
            if not torch.is_tensor(p) or id(p) not in ids:
                raise NotImplementedError("adjoint_params may only hold parameters of the ODENet being integrated "
                                          "(gene_multipliers and the weights / biases of its three linear layers)")
            if id(p) in seen:
                raise NotImplementedError("adjoint_params holds the same parameter twice")
            seen.add(id(p))
    mask = 0
    for i, p in enumerate(params):
        if p.requires_grad and any(p is c for c in chosen):
            mask |= 1 << i
    return params, mask


def _adjoint_norm(adjoint_options):
    """Take ``norm`` out of the adjoint options: the remaining options and the norm's bit of the adjoint mask
    (NORM_SEMINORM for ``"seminorm"``, 0 when no norm is given)."""
    if adjoint_options is None or "norm" not in adjoint_options:
        return adjoint_options, 0
    opts = dict(adjoint_options)
    norm = opts.pop("norm")
    if not (isinstance(norm, str) and norm == "seminorm"):
        raise NotImplementedError('adjoint_options["norm"] = {!r} is not supported: the error norm is evaluated on the '
                                  'device, and only "seminorm" (the mixed norm without the parameter block) is '
                                  'implemented there'.format(norm))
    return opts, NORM_SEMINORM


def odeint_adjoint(func, y0, t, rtol=1e-7, atol=1e-9, method=None, options=None, adjoint_rtol=None,
                   adjoint_atol=None, adjoint_method=None, adjoint_options=None, adjoint_params=None):
    """adjoint.py:165-204: same as ``odeint`` but differentiable w.r.t. y0 and the ODENet parameters through the
    continuous adjoint, solved backwards with the forward method / tolerances unless overridden.
    ``adjoint_options=dict(norm="seminorm")`` measures the dopri5 backward's error without the parameter cotangents
    (Kidger, Chen & Lyons, 2021), in the initial step and in every error ratio."""
    if adjoint_params is None and not isinstance(func, nn.Module):
        raise ValueError('func must be an instance of nn.Module to specify the adjoint parameters; alternatively they '
                         'can be specified explicitly via the `adjoint_params` argument. If there are no parameters '
                         'then it is allowable to set `adjoint_params=()`.')
    if adjoint_rtol is None:
        adjoint_rtol = rtol
    if adjoint_atol is None:
        adjoint_atol = atol
    if adjoint_method is None:
        adjoint_method = method
    adjoint_options, norm_bit = _adjoint_norm(adjoint_options)
    if adjoint_options is None:
        adjoint_options = {k: v for k, v in options.items() if k != "norm"} if options is not None else {}
    same = (adjoint_rtol is rtol and adjoint_atol is atol and adjoint_method is method and not adjoint_options
            and not options)
    tl, t_is_f32, rev, rtol, atol, method, max_steps = _normalise(func, y0, t, rtol, atol, method, options)
    step, ctl = _step_size(method, options), _step_control(method, options)
    if same:
        a_rtol, a_atol, a_method, a_max, a_step, a_ctl = rtol, atol, method, max_steps, step, ctl
    else:
        _, _, _, a_rtol, a_atol, a_method, a_max = _normalise(func, y0, t, adjoint_rtol, adjoint_atol, adjoint_method,
                                                              adjoint_options)
        a_step, a_ctl = _step_size(a_method, adjoint_options), _step_control(a_method, adjoint_options)
    if rev:
        raise NotImplementedError("odeint_adjoint with decreasing t is not part of the PHOENIX path")
    params, mask = _adjoint_mask(func, adjoint_params)
    return OdeintAdjointMethod.apply(func, tl, t_is_f32, _with_control((method, step), ctl), rtol, atol, max_steps,
                                     _with_control((a_method, a_rtol, a_atol, a_max, mask | norm_bit, a_step), a_ctl),
                                     y0, *params)


class OdeintAdjointManyMethod(torch.autograd.Function):
    """N independent ``OdeintAdjointMethod`` problems behind one autograd node (engine.solve_*_many)."""

    @staticmethod
    def forward(ctx, func, t_rows, t_is_f32, fwd, rtol, atol, max_steps, adj, y0, *adjoint_params):
        ctx.func, ctx.t_rows, ctx.t_is_f32, ctx.adj = func, t_rows, t_is_f32, adj
        with torch.no_grad():
            y = engine.solve_forward_many(func, y0, t_rows, t_is_f32, fwd[0], rtol, atol, max_steps, **_stepped(fwd[1]),
                                          **_controlled(fwd, 2))
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, grad_y):
        (y,) = ctx.saved_tensors
        a_method, a_rtol, a_atol, a_max, mask = ctx.adj[:5]
        if not mask & PARAMS_ALL and not ctx.needs_input_grad[8]:
            return (None,) * (9 + len(ctx.needs_input_grad[9:]))
        with torch.no_grad():
            adj_y0, grads = engine.solve_adjoint_many(ctx.func, ctx.t_rows, ctx.t_is_f32, a_method, a_rtol, a_atol,
                                                      a_max, y, grad_y, **_masked(mask), **_stepped(ctx.adj[5]),
                                                      **_controlled(ctx.adj, 6))
        return _grads_out(ctx, adj_y0, grads, mask)


def odeint_adjoint_many(func, y0, t, rtol=1e-7, atol=1e-9, method=None, options=None, adjoint_params=None,
                        adjoint_options=None):
    """The per-sample loop of the reference's ``training_step`` (train_insilico.py:128-130,
    ``[odeint(odenet, batch_point, time_points, method=method)[1] for ...]``) as ONE call: ``y0`` is ``[N, *S, G]``
    (N independent initial states), ``t`` is ``[N, T]`` (each sample's own times, increasing) and the result is
    ``[N, T, *S, G]`` with ``result[i] == odeint_adjoint(func, y0[i], t[i], ...)`` bit for bit: every sample is still
    its own solve with its own step controller (NOT the global-norm batched call).  Gradients flow to ``y0`` and to the
    ODENet parameters of ``adjoint_params`` that require grad (default: all six; summed over the samples) through one
    autograd node.  ``adjoint_options`` as in ``odeint_adjoint`` (default: the forward options without ``norm``).  No
    reference counterpart: opt-in."""
    assert torch.is_tensor(t) and t.ndimension() == 2, "t must be a [N, T] tensor of per-sample times"
    assert torch.is_tensor(y0) and y0.shape[0] == t.shape[0], "y0 and t must hold the same number of samples"
    if y0.shape[0] == 0:
        raise ValueError("odeint_adjoint_many needs at least one sample")
    t_is_f32 = t.dtype != torch.float64
    rows = t.tolist()
    tl0, _, rev, rtol_f, atol_f, method, max_steps = _normalise(func, y0[0], t[0], rtol, atol, method, options)
    for r in rows:
        assert all(b > a for a, b in zip(r, r[1:])), 't must be strictly increasing for every sample'
    if rev:
        raise NotImplementedError("odeint_adjoint_many with decreasing t is not part of the PHOENIX path")
    step, ctl = _step_size(method, options), _step_control(method, options)
    adjoint_options, norm_bit = _adjoint_norm(adjoint_options)
    a_max, a_step, a_ctl = max_steps, step, ctl
    if adjoint_options is not None:
        a_max = _normalise(func, y0[0], t[0], rtol, atol, method, adjoint_options)[6]
        a_step, a_ctl = _step_size(method, adjoint_options), _step_control(method, adjoint_options)
    params, mask = _adjoint_mask(func, adjoint_params)
    return OdeintAdjointManyMethod.apply(func, rows, t_is_f32, _with_control((method, step), ctl), rtol_f, atol_f,
                                         max_steps,
                                         _with_control((method, rtol_f, atol_f, a_max, mask | norm_bit, a_step), a_ctl),
                                         y0, *params)
