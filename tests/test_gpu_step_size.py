"""Fixed-grid solves on a step grid: ``options=dict(step_size=h)`` for euler, midpoint and rk4, forward and adjoint.

torchdiffeq 0.1.1's ``FixedGridODESolver`` (solvers.py:48-50, 77-103) steps on the grid ``arange(0, ceil((t[-1] - t[0]) / h
+ 1)) * h + t[0]`` (last point clamped to t[-1], in the dtype of t) and interpolates linearly the output times that fall
inside a step; the state is not restarted at the output times.  The adjoint's backward integrates every output interval
on a grid of its own over the negated times.  The oracle below extends ``oracle/phoenix_oracle.py`` with exactly that;
with no step size it is the oracle itself.  CPU tests pin the oracle, the host grids and the option parsing; GPU tests run
every engine (resident, resident many, rows at 4 / 2 / 1 rows per pass, streaming)."""
import math

import pytest
import torch

import phoenix_b200 as pbm
from phoenix_b200 import engine as E
from phoenix_b200.torchdiffeq import _api
from oracle import phoenix_oracle as O
from golden_util import rel_l2
from test_gpu_placements import make_net

NAMES = O.PARAM_ORDER
METHODS = ("euler", "midpoint", "rk4")


# ---- oracle (CPU) ----------------------------------------------------------------------------------------------------------
def oracle_grid(t, step_size):
    """solvers.py:48-50 (``_grid_constructor_from_step_size``) and the assertion of solvers.py:77."""
    if step_size is None:
        return t
    niters = torch.ceil((t[-1] - t[0]) / step_size + 1).item()
    grid = torch.arange(0, niters, dtype=t.dtype, device=t.device) * step_size + t[0]
    if grid[-1] > t[-1]:
        grid[-1] = t[-1]
    assert grid[0] == t[0] and grid[-1] == t[-1]
    return grid


def _step(method, f, t0, dt, y):
    """dy of one step (fixed_grid.py:13-14, 24-27; rk4 = 3/8 rule rk_common.py:96-103), as O._solve_fixed forms it."""
    if method == "euler":
        return dt * f(t0, y)
    if method == "midpoint":
        half = 0.5 * dt
        return dt * f(t0 + half, y + f(t0, y) * half)
    k1 = f(t0, y)
    k2 = f(t0 + dt / 3, y + dt * k1 * (1 / 3))
    k3 = f(t0 + dt * (2 / 3), y + dt * (k2 - k1 * (1 / 3)))
    k4 = f(t0 + dt, y + dt * (k1 - k2 + k3))
    return (k1 + 3 * (k2 + k3) + k4) * dt * 0.125


def solve_fixed_grid(func, y0, t, method, log, step_size, where=None):
    """solvers.py:77-103 on the grid of ``step_size`` (None: grid = t).  ``where`` (a list) receives, per output time
    j >= 1, (step index, slope or None for an exact hit)."""
    grid = oracle_grid(t, step_size)
    out = torch.empty(len(t), *y0.shape, dtype=y0.dtype)
    out[0] = y0

    def f(tt, yy):
        log.nfe += 1
        return func(tt, yy)

    j, y = 1, y0
    for k, (t0, t1) in enumerate(zip(grid[:-1], grid[1:])):
        y1 = y + _step(method, f, t0, t1 - t0, y)
        while j < len(t) and t1 >= t[j]:
            if t[j] == t0:
                out[j] = y
                slope = 0.0
            elif t[j] == t1:
                out[j] = y1
                slope = None
            else:
                slope = (t[j] - t0) / (t1 - t0)
                out[j] = y + slope * (y1 - y)
            if where is not None:
                where.append((k, slope))
            j += 1
        y = y1
    return out


def odeint_ss(w, y0, t, method, step_size=None, where=None):
    """``O.odeint`` for the fixed-grid methods with ``options=dict(step_size=...)``; returns (y, StepLog)."""
    log = O.StepLog([])
    sign = 1.0
    if bool((t[1:] < t[:-1]).all()):
        sign, t = -1.0, -t
    func = (lambda tt, yy: O.rhs(w, yy)) if sign > 0 else (lambda tt, yy: -O.rhs(w, yy))
    with torch.no_grad():
        y = solve_fixed_grid(func, y0, t, method, log, step_size, where)
    return y, log


def adjoint_backward_ss(w, t, y, grad_y, method, step_size=None):
    """``O.adjoint_backward`` with ``adjoint_options=dict(step_size=...)``: every interval [t[i-1], t[i]] is integrated
    on its own grid over ``-t[i-1:i+1].flip(0)``.  Returns (adj_y0, [6 grads], StepLog)."""
    log = O.StepLog([])
    shape = y.shape[1:]
    N = y[0].numel()
    params = w.as_list()
    psz = [p.numel() for p in params]

    def aug_reversed(tt, z):
        f, ybar, pbar = O.rhs_vjp(w, z[1:1 + N].reshape(shape), -z[1 + N:1 + 2 * N].reshape(shape))
        return -torch.cat([torch.zeros(1, dtype=z.dtype), f.reshape(-1), ybar.reshape(-1)] + [p.reshape(-1) for p in pbar])

    with torch.no_grad():
        adj_y = grad_y[-1].clone()
        adj_p = torch.zeros(sum(psz), dtype=y.dtype)
        cur_y = y[-1]
        for i in range(len(t) - 1, 0, -1):
            z0 = torch.cat([torch.zeros(1, dtype=y.dtype), cur_y.reshape(-1), adj_y.reshape(-1), adj_p])
            z = solve_fixed_grid(aug_reversed, z0, -t[i - 1:i + 1].flip(0), method, log, step_size)[1]
            adj_p = z[1 + 2 * N:]
            cur_y = y[i - 1]
            adj_y = z[1 + N:1 + 2 * N].reshape(shape) + grad_y[i - 1]
        grads, lo = [], 0
        for p, n in zip(params, psz):
            grads.append(adj_p[lo:lo + n].reshape(p.shape))
            lo += n
    return adj_y, grads, log


def _small(method="rk4", T=3, dtype=torch.float64):
    w = O.make_weights(37, 5, 3, dense=True, neg_mult_frac=0.2)
    y0 = torch.rand(1, 37, generator=torch.Generator().manual_seed(4))
    t = torch.tensor([0.0, 0.45, 1.0, 1.3][:T], dtype=dtype)
    return w, y0, t


@pytest.mark.parametrize("method", METHODS)
def test_oracle_without_step_size_is_the_oracle(method):
    w, y0, t = _small(method)
    y_ref, log_ref = O.odeint(w, y0, t, method=method)
    y, log = odeint_ss(w, y0, t, method)
    assert torch.equal(y, y_ref) and log.nfe == log_ref.nfe
    gy = torch.rand_like(y, generator=torch.Generator().manual_seed(5))
    a_ref, g_ref, _ = O.adjoint_backward(w, t, y, gy, method=method)
    a, g, _ = adjoint_backward_ss(w, t, y, gy, method)
    assert torch.equal(a, a_ref) and all(torch.equal(x, r) for x, r in zip(g, g_ref))
    # a grid that is t itself (one interval, step >= its span) is the same solve
    t2 = t[:2]
    assert torch.equal(odeint_ss(w, y0, t2, method, 2.0)[0], O.odeint(w, y0, t2, method=method)[0])


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_hand_checked_grids(dtype):
    g = oracle_grid(torch.tensor([0.0, 1.0], dtype=dtype), 0.3)
    assert g.dtype == dtype and len(g) == 5 and g[0] == 0 and g[-1] == 1.0
    assert torch.allclose(g, torch.tensor([0.0, 0.3, 0.6, 0.9, 1.0], dtype=dtype))
    assert torch.equal(oracle_grid(torch.tensor([0.0, 1.0], dtype=dtype), 0.25),
                       torch.tensor([0.0, 0.25, 0.5, 0.75, 1.0], dtype=dtype))   # an exact multiple: no clamp
    for t in ([0.0, 1.0], [0.5, 0.8], [-1.3, -0.2], [0.0, 0.9]):
        for h in (0.3, 0.25, 0.07, 5.0):
            tt = torch.tensor(t, dtype=dtype)
            try:
                ref = oracle_grid(tt, h)
            except AssertionError:
                with pytest.raises(AssertionError):
                    E.fixed_grid(tt, h)
                continue
            assert torch.equal(E.fixed_grid(tt, h), ref)


@pytest.mark.parametrize("dtype,t1,h", [(torch.float64, 0.9, 0.3), (torch.float32, 2.7, 0.9)])
def test_end_point_assertion(dtype, t1, h):
    """Rounding leaves the last grid point short of t[-1]: the reference's own assertion, on both sides."""
    t = torch.tensor([0.0, t1], dtype=dtype)
    with pytest.raises(AssertionError):
        oracle_grid(t, h)
    with pytest.raises(AssertionError):
        E.forward_grid(t.tolist(), dtype == torch.float32, h)
    with pytest.raises(AssertionError):
        E.adjoint_grid(t.tolist(), dtype == torch.float32, h)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("method", METHODS)
def test_outputs_inside_a_step(method, dtype):
    """Output times inside a step (0.45: slope 1/2), on a grid point (0.6 in float32), several in one step (0.61, 0.65,
    0.7 in the step from 0.6): each is y + s (y1 - y) of the states at the step's ends -- the solve on the grid points
    themselves -- and the state goes on from the grid point, not from the output."""
    w = O.make_weights(37, 5, 3, dense=True, neg_mult_frac=0.2)
    y0 = torch.rand(1, 37, generator=torch.Generator().manual_seed(4))
    t = torch.tensor([0.0, 0.45, 0.6, 0.61, 0.65, 0.7, 1.0], dtype=dtype)
    where = []
    y, log = odeint_ss(w, y0, t, method, 0.3, where)
    grid = oracle_grid(t, 0.3)
    ygrid, _ = odeint_ss(w, y0, grid, method)
    assert log.nfe == {"euler": 1, "midpoint": 2, "rk4": 4}[method] * (len(grid) - 1)
    assert len(where) == len(t) - 1 and [k for k, _ in where] == [1, 1, 2, 2, 2, 3]
    for j, (k, s) in enumerate(where, start=1):
        if s is None:
            assert torch.equal(y[j], ygrid[k + 1])
        else:
            assert torch.equal(y[j], ygrid[k] + s * (ygrid[k + 1] - ygrid[k]))
    assert torch.equal(y[-1], ygrid[-1])


def _where_arrays(t, h):
    where = []
    w = O.make_weights(7, 2, 1)
    odeint_ss(w, torch.rand(1, 7), t, "euler", h, where)
    k = torch.tensor([q for q, _ in where], dtype=torch.int32)
    s = torch.tensor([-1.0 if q is None else float(q) for _, q in where], dtype=torch.float32)
    return k, s


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_host_grids_match_the_oracle(dtype):
    """engine.forward_grid / adjoint_grid (what the kernels get) against the oracle's grid, step map and slopes, and the
    backward grids of every interval; decreasing t is negated first, as the reference does."""
    cases = [([0.0, 0.45, 0.6, 0.65, 1.0], 0.3), ([0.2, 0.7, 1.9], 0.25), ([0.0, 0.1], 1.0), ([3.0, 1.5, 0.0], 0.4),
             ([0.0, 5.0, 10.0, 20.0], 1.0), ([0.1, 0.2, 0.3], 0.0137)]
    for tl, h in cases:
        t = torch.tensor(tl, dtype=dtype)
        ts = -t if tl[1] < tl[0] else t
        dt, k, s = E.forward_grid(ts.tolist(), dtype == torch.float32, h)
        g = oracle_grid(ts, h)
        assert torch.equal(dt, (g[1:] - g[:-1]).float())
        kr, sr = _where_arrays(ts, h)
        assert torch.equal(k, kr) and torch.equal(s, sr), (tl, h)
        if tl[1] < tl[0]:
            continue
        dts, counts = E.adjoint_grid(t.tolist(), dtype == torch.float32, h)
        ref = []
        for i in range(1, len(t)):
            gi = oracle_grid(-t[i - 1:i + 1].flip(0), h)
            ref.append((gi[1:] - gi[:-1]).float())
        assert counts == [len(r) for r in ref] and torch.equal(dts, torch.cat(ref))


# ---- option parsing (CPU) ----------------------------------------------------------------------------------------------------
def _cpu_net():
    torch.manual_seed(0)
    return pbm.ODENet("cpu", 12, neurons=4)


def _captured(monkeypatch, many, method="rk4", **kw):
    """(fwd, adj) an entry point hands its autograd node: fwd = (method, step_size), adj[5] = the backward step size."""
    got = {}

    def fake_apply(*args):
        got["fwd"], got["adj"] = args[3], args[7]
        return None

    cls = _api.OdeintAdjointManyMethod if many else _api.OdeintAdjointMethod
    monkeypatch.setattr(cls, "apply", fake_apply)
    net = _cpu_net()
    y0 = torch.rand(1, 12)
    t = torch.tensor([0.0, 1.0])
    if many:
        pbm.odeint_adjoint_many(net, y0.unsqueeze(0), t.unsqueeze(0), method=method, **kw)
    else:
        pbm.odeint_adjoint(net, y0, t, method=method, **kw)
    return got["fwd"], got["adj"]


@pytest.mark.parametrize("many", [False, True])
def test_adjoint_inherits_the_step_size(monkeypatch, many):
    assert _captured(monkeypatch, many) == (("rk4", None), ("rk4", 1e-7, 1e-9, 2 ** 31 - 1, 0x3F, None))
    fwd, adj = _captured(monkeypatch, many, options=dict(step_size=0.25))
    assert fwd == ("rk4", 0.25) and adj[5] == 0.25
    fwd, adj = _captured(monkeypatch, many, options=dict(step_size=0.25), adjoint_options=dict(step_size=0.1))
    assert fwd == ("rk4", 0.25) and adj[5] == 0.1
    fwd, adj = _captured(monkeypatch, many, options=dict(step_size=0.25), adjoint_options={})
    assert fwd == ("rk4", 0.25) and adj[5] is None
    fwd, adj = _captured(monkeypatch, many, adjoint_options=dict(step_size=0.5, norm="seminorm"))
    assert fwd == ("rk4", None) and adj[5] == 0.5 and adj[4] == 0x7F
    fwd, adj = _captured(monkeypatch, many, options=dict(step_size=torch.tensor(0.5)))
    assert fwd == ("rk4", (0.5, torch.float32)) and adj[5] == (0.5, torch.float32)
    fwd, adj = _captured(monkeypatch, many, options=dict(step_size=torch.tensor(0.1, dtype=torch.float64)))
    assert fwd == ("rk4", (0.1, torch.float64)) and adj[5] == fwd[1]


# float32 t = [0, 1.1] with a float64 0-dim tensor step 0.1: the reference divides the span in float64 (both operands are
# 0-dim) and gets one grid point more than with the Python float 0.1, so its last step has zero length
T_F32 = [0.0, 1.1]
H_F64 = torch.tensor(0.1, dtype=torch.float64)


def test_tensor_step_size_keeps_its_dtype():
    t = torch.tensor(T_F32, dtype=torch.float32)
    ref = oracle_grid(t, H_F64)
    assert len(ref) == len(oracle_grid(t, 0.1)) + 1 and ref[-1] == ref[-2]
    step = _api._stepped(_api._step_size("rk4", dict(step_size=H_F64)))["step_size"]
    assert step.dtype == torch.float64 and torch.equal(step, H_F64)
    assert torch.equal(E.fixed_grid(t, step), ref)
    dt, k, s = E.forward_grid(T_F32, True, step)
    assert torch.equal(dt, (ref[1:] - ref[:-1]).float()) and dt[-1] == 0
    kr, sr = _where_arrays(t, H_F64)
    assert torch.equal(k, kr) and torch.equal(s, sr)


def _entry_points():
    net = _cpu_net()
    y0 = torch.rand(1, 12)
    t = torch.tensor([0.0, 1.0])
    return {
        "odeint": lambda **kw: pbm.odeint(net, y0, t, **kw),
        "odeint_adjoint": lambda **kw: pbm.odeint_adjoint(net, y0, t, **kw),
        "odeint_adjoint_many": lambda **kw: pbm.odeint_adjoint_many(net, y0.unsqueeze(0), t.unsqueeze(0), **kw),
    }


@pytest.mark.parametrize("entry", ["odeint", "odeint_adjoint", "odeint_adjoint_many"])
def test_step_size_refusals(entry):
    solve = _entry_points()[entry]
    for method in (None, "dopri5"):
        with pytest.raises(NotImplementedError):
            solve(method=method, options=dict(step_size=0.1))
    for method in ("dopri5", "rk4"):
        with pytest.raises(NotImplementedError, match="grid_constructor"):
            solve(method=method, options=dict(grid_constructor=lambda f, y, t: t))
    with pytest.raises(NotImplementedError, match="0-dimensional"):
        solve(method="rk4", options=dict(step_size=torch.tensor([0.1])))
    for bad in (0.0, -0.1, float("inf"), float("nan"), torch.tensor(-1.0)):
        with pytest.raises(ValueError, match="step_size"):
            solve(method="rk4", options=dict(step_size=bad))
    if entry != "odeint":
        with pytest.raises(ValueError, match="step_size"):
            solve(method="rk4", adjoint_options=dict(step_size=0.0))
        with pytest.raises(NotImplementedError, match="grid_constructor"):
            solve(method="rk4", adjoint_options=dict(grid_constructor=lambda f, y, t: t))


class _Ctx:
    def __init__(self, **kw):
        self.__dict__.update(kw)


def test_deferred_group_key_includes_the_step_size(monkeypatch):
    monkeypatch.setattr(_api, "DEFER_ADJOINT", True)
    net = _cpu_net()
    y0 = torch.rand(1, 12)
    keys = []
    for h in (None, 0.1, 0.2, 0.1):
        ctx = _Ctx(needs_input_grad=(False,) * 9 + (True,) * 6)
        _api._register_node(ctx, net, y0, [0.0, 1.0], True, ("rk4", 1e-7, 1e-9, 100, 0x3F, h))
        keys.append(ctx.group)
    assert len({keys[0], keys[1], keys[2]}) == 3 and keys[1] == keys[3]


# ---- GPU -----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pb():
    pbm.set_sync_errors(True)
    yield pbm
    pbm.engine.FORCE_ENGINE = None


def _weights(G, H, seed):
    w = O.make_weights(G, H, seed, dense=True, neg_mult_frac=0.2)
    if G > 1000:
        w.Wp.mul_((1000.0 / G) ** 0.5)
        w.Ws.mul_((1000.0 / G) ** 0.5)
    return w


# (engine, G, H, y0 shape, many).  many: odeint_adjoint_many, N problems of the given per-problem shape.
ENGINES = [
    ("resident", 350, 40, (1, 350), False),
    ("resident", 350, 40, (3, 2, 350), True),    # phx_solve_*_many shapes
    ("rows", 690, 200, (5, 1, 690), True),       # 4 rows per pass
    ("rows", 13000, 129, (3, 1, 13000), True),   # 2 rows per pass
    ("rows", 16000, 100, (3, 1, 16000), True),   # 1 row per pass
    ("stream", 350, 40, (6, 350), False),
]


def _eid(e):
    return "%s-%dx%d-%s%s" % (e[0], e[1], e[2], "x".join(map(str, e[3])), "-many" if e[4] else "")


def _times(many, n, base, dtype=torch.float64):
    """Output times: one row of ``base``; with ``many``, problem i shifted by i / 7 and its span stretched by
    (1 + i / 3), so that rows of one pass take different numbers of steps."""
    base = torch.tensor(base, dtype=torch.float64)
    if not many:
        return base.to(dtype)
    rows = [(base - base[0]) * (1 + i / 3.0) + base[0] + i / 7.0 for i in range(n)]
    return torch.stack(rows).to(dtype)


def _run(pb, net, y0, t, target, method, engine, many, options=None, adjoint_options=None):
    """Forward + backward through odeint_adjoint(_many) on the GPU: y, adj_y0, the six .grad."""
    saved = pb.engine.FORCE_ENGINE
    pb.engine.FORCE_ENGINE = engine
    try:
        net.zero_grad(set_to_none=True)
        y0g = y0.cuda().requires_grad_(True)
        solve = pb.odeint_adjoint_many if many else pb.odeint_adjoint
        y = solve(net, y0g, t, method=method, options=options, adjoint_options=adjoint_options)
        ys = y[:, 1:] if many else y[1:]
        ((ys - target.cuda()) ** 2).sum().backward()
        return y.detach().cpu(), y0g.grad.cpu(), [p.grad.detach().cpu().clone() for p in net.parameters()]
    finally:
        pb.engine.FORCE_ENGINE = saved


def _problem(e, base, seed, dtype=torch.float64):
    engine, G, H, shape, many = e
    w = _weights(G, H, seed)
    gen = torch.Generator().manual_seed(seed + 1)
    y0 = torch.rand(*shape, generator=gen)
    t = _times(many, shape[0], base, dtype)
    target = torch.rand(*((shape[0], len(base) - 1) + shape[1:] if many else (len(base) - 1,) + shape), generator=gen)
    return w, y0, t, target


def _same(a, b):
    return torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and all(torch.equal(x, z) for x, z in zip(a[2], b[2]))


@pytest.mark.gpu
@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("e", ENGINES, ids=[_eid(e) for e in ENGINES])
def test_grid_equal_to_t_is_bit_identical(pb, e, method):
    """T = 2 with step_size >= the span: the grid is t, so forward and backward give today's bits; and a step size
    larger than every interval, given to the backward only, of a multi-interval t: every backward interval is one step."""
    w, y0, t, target = _problem(e, (0.0, 0.1), 31)
    net = make_net(pb, w)
    ref = _run(pb, net, y0, t, target, method, e[0], e[4])
    got = _run(pb, net, y0, t, target, method, e[0], e[4], options=dict(step_size=0.5))
    assert _same(got, ref)
    w, y0, t, target = _problem(e, (0.0, 0.05, 0.1), 32)
    net = make_net(pb, w)
    ref = _run(pb, net, y0, t, target, method, e[0], e[4])
    got = _run(pb, net, y0, t, target, method, e[0], e[4], adjoint_options=dict(step_size=1.0))
    assert _same(got, ref)


def _oracle_fwd(w, y0, t, method, h, many):
    if many:
        outs = [odeint_ss(w, y0[i], t[i], method, h) for i in range(y0.shape[0])]
        return torch.stack([o[0] for o in outs]), [o[1].nfe for o in outs]
    y, log = odeint_ss(w, y0, t, method, h)
    return y, [log.nfe]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("e", ENGINES, ids=[_eid(e) for e in ENGINES])
def test_forward_against_oracle(pb, e, method, dtype):
    """Output times inside steps, increasing t (every engine; many problems of different spans) and decreasing t (the
    one-problem calls), float32 and float64 t: relative L2 <= 1e-5 against the fp32 oracle, and status n_rhs equals the
    oracle's number of evaluations."""
    engine, G, H, shape, many = e
    base = (0.0, 0.013, 0.05, 0.071, 0.1)
    w, y0, t, _ = _problem(e, base, 47, dtype)
    net = make_net(pb, w)
    h = 0.0175   # (0.02 would miss t[-1] on the float32 grid: the reference's assertion)
    saved = pb.engine.FORCE_ENGINE
    pb.engine.FORCE_ENGINE = engine
    try:
        cases = [t] if many else [t, t.flip(0)]
        for tt in cases:
            if many:
                y = pb.odeint_adjoint_many(net, y0.cuda(), tt, method=method, options=dict(step_size=h)).detach().cpu()
            else:
                y = pb.odeint(net, y0.cuda(), tt, method=method, options=dict(step_size=h)).cpu()
                n_rhs = pb.engine.last_status()["n_rhs"]
            y_ref, nfe = _oracle_fwd(w, y0, tt, method, h, many)
            assert rel_l2(y, y_ref) <= 1e-5, (_eid(e), method, dtype, rel_l2(y, y_ref))
            if not many:
                assert n_rhs == nfe[0], (n_rhs, nfe)
    finally:
        pb.engine.FORCE_ENGINE = saved


def _oracle_adj(w, y0, t, target, method, h, many):
    probs = [(y0[i], t[i], target[i]) for i in range(y0.shape[0])] if many else [(y0, t, target)]
    ys, adys, gsum = [], [], None
    for y0i, ti, tgi in probs:
        yr, _ = odeint_ss(w, y0i, ti, method, h)
        gy = torch.zeros_like(yr)
        gy[1:] = 2.0 * (yr[1:] - tgi)
        ar, gr, _ = adjoint_backward_ss(w, ti, yr, gy, method, h)
        ys.append(yr)
        adys.append(ar)
        gsum = gr if gsum is None else [a + b for a, b in zip(gsum, gr)]
    return (torch.stack(ys) if many else ys[0]), (torch.stack(adys) if many else adys[0]), gsum


@pytest.mark.gpu
@pytest.mark.parametrize("T", [2, 3])
@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("e", ENGINES, ids=[_eid(e) for e in ENGINES])
def test_adjoint_against_oracle(pb, e, method, T):
    """y, adj_y0 and the six gradients (relative L2 <= 1e-5) against the oracle's backward on the per-interval grids;
    the rows passes hold problems of different spans, so their rows take different numbers of steps in every interval
    (with T = 3 the rows kernel also carries y and adj_y from step to step inside an interval and adj_y across them)."""
    base = (0.0, 0.07, 0.1)[:T]
    w, y0, t, target = _problem(e, base, 53)
    net = make_net(pb, w)
    h = 0.02
    y, ady, grads = _run(pb, net, y0, t, target, method, e[0], e[4], options=dict(step_size=h))
    y_ref, ady_ref, g_ref = _oracle_adj(w, y0, t, target, method, h, e[4])
    assert rel_l2(y, y_ref) <= 1e-5
    assert rel_l2(ady, ady_ref) <= 1e-5, (_eid(e), rel_l2(ady, ady_ref))
    for i in range(6):
        assert rel_l2(grads[i], g_ref[i]) <= 1e-5, (_eid(e), NAMES[i], rel_l2(grads[i], g_ref[i]))


@pytest.mark.gpu
@pytest.mark.parametrize("method", METHODS)
def test_rows_property_with_uneven_step_counts(pb, method):
    """A problem's y and adj_y0 are the same bits alone and as a row of a pass beside rows with more and fewer steps."""
    G, H = 690, 200
    w = _weights(G, H, 61)
    net = make_net(pb, w)
    gen = torch.Generator().manual_seed(62)
    y0 = torch.rand(4, 1, G, generator=gen)
    t = torch.tensor([[0.0, 0.1], [0.3, 0.33], [0.0, 0.25], [1.0, 1.05]], dtype=torch.float64)
    target = torch.rand(4, 1, 1, G, generator=gen)
    opts = dict(step_size=0.02)
    together = _run(pb, net, y0, t, target, method, "rows", True, options=opts)
    for i in range(4):
        alone = _run(pb, net, y0[i:i + 1], t[i:i + 1], target[i:i + 1], method, "rows", True, options=opts)
        assert torch.equal(alone[0][0], together[0][i]) and torch.equal(alone[1][0], together[1][i]), (method, i)


@pytest.mark.gpu
@pytest.mark.parametrize("method", METHODS)
def test_per_sample_loop_with_step_size_matches_many(pb, monkeypatch, method):
    """The literal loop of training_step with a step size: under SINGLE_CALL_ENGINE="rows" the deferred backward gives
    odeint_adjoint_many's gradients bit for bit; with the default engine choice, to rounding."""
    G, H, N = 690, 40, 6
    w = O.make_weights(G, H, 21, dense=True, neg_mult_frac=0.2)
    gen = torch.Generator().manual_seed(22)
    y0 = torch.rand(N, 1, G, generator=gen)
    t = torch.rand(N, 1, generator=gen, dtype=torch.float64) + torch.tensor([0.0, 0.1], dtype=torch.float64)
    target = torch.rand(N, 1, G, generator=gen)
    net = make_net(pb, w)
    params = list(net.parameters())
    opts = dict(step_size=0.03)
    net.zero_grad(set_to_none=True)
    y = pb.odeint_adjoint_many(net, y0.cuda(), t, method=method, options=opts)
    torch.mean((y[:, 1] - target.cuda()) ** 2).backward()
    many = [p.grad.clone() for p in params]
    for single, exact in (("rows", True), (pb.engine.SINGLE_CALL_ENGINE, False)):
        monkeypatch.setattr(pb.engine, "SINGLE_CALL_ENGINE", single)
        net.zero_grad(set_to_none=True)
        preds = [pb.odeint_adjoint(net, y0[i].cuda(), t[i], method=method, options=opts)[1] for i in range(N)]
        torch.mean((torch.stack(preds) - target.cuda()) ** 2).backward()
        for i in range(6):
            if exact:
                assert torch.equal(params[i].grad, many[i]), (method, NAMES[i])
            else:
                assert rel_l2(params[i].grad.cpu(), many[i].cpu()) <= 1e-5, (method, NAMES[i])


@pytest.mark.gpu
def test_steps_are_really_taken(pb):
    """A yeast-like output spacing (dt = 10) with a 350 x 40 model: rk4 with step_size = 1 is much closer to a float64
    dopri5 solve (rtol 1e-10) than one rk4 step per interval.  The two errors are printed."""
    w = O.make_weights(350, 40, 71, dense=True, neg_mult_frac=0.2)
    w.Wp.mul_(0.3)
    w.Ws.mul_(0.3)
    net = make_net(pb, w)
    y0 = torch.rand(1, 350, generator=torch.Generator().manual_seed(72))
    t = torch.tensor([0.0, 10.0, 20.0], dtype=torch.float64)
    wd = O.Weights(*[p.double() for p in w.as_list()])
    y64, _ = O.odeint(wd, y0.double(), t, method="dopri5", rtol=1e-10, atol=1e-12)
    one = pb.odeint(net, y0.cuda(), t, method="rk4").cpu()
    fine = pb.odeint(net, y0.cuda(), t, method="rk4", options=dict(step_size=1.0)).cpu()
    e_one, e_fine = rel_l2(one[1:], y64[1:].float()), rel_l2(fine[1:], y64[1:].float())
    if not math.isfinite(e_one):   # one 3/8-rule step over dt = 10 may leave the range of float32 altogether
        e_one = float("inf")
    print("rk4 against float64 dopri5, relative L2: one step per interval %.3e, step_size=1 %.3e" % (e_one, e_fine))
    assert e_fine < 0.1 * e_one and e_fine < 1e-4, (e_one, e_fine)


TENSOR_ENGINES = [("resident", 350, 40, (1, 350), False), ("rows", 690, 200, (3, 1, 690), True),
                  ("stream", 350, 40, (6, 350), False)]


@pytest.mark.gpu
@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("e", TENSOR_ENGINES, ids=[_eid(e) for e in TENSOR_ENGINES])
def test_float64_tensor_step_on_float32_t(pb, e, method):
    """float32 t and a float64 tensor step size: the grid of the reference (one point more than with the float, a last
    step of zero length) -- forward (n_rhs = the oracle's evaluations) and backward against the oracle."""
    engine, G, H, shape, many = e
    w = _weights(G, H, 81)
    net = make_net(pb, w)
    gen = torch.Generator().manual_seed(82)
    y0 = torch.rand(*shape, generator=gen)
    t = torch.tensor(T_F32, dtype=torch.float32)
    if many:
        t = t.repeat(shape[0], 1)
        target = torch.rand(shape[0], 1, *shape[1:], generator=gen)
    else:
        target = torch.rand(1, *shape, generator=gen)
    opts = dict(step_size=H_F64)
    if not many:
        saved = pb.engine.FORCE_ENGINE
        pb.engine.FORCE_ENGINE = engine
        try:
            pb.odeint(net, y0.cuda(), t, method=method, options=opts)
            n_rhs = pb.engine.last_status()["n_rhs"]
        finally:
            pb.engine.FORCE_ENGINE = saved
        assert n_rhs == odeint_ss(w, y0, t, method, H_F64)[1].nfe
    y, ady, grads = _run(pb, net, y0, t, target, method, engine, many, options=opts)
    y_ref, ady_ref, g_ref = _oracle_adj(w, y0, t, target, method, H_F64, many)
    assert rel_l2(y, y_ref) <= 1e-5 and rel_l2(ady, ady_ref) <= 1e-5, (rel_l2(y, y_ref), rel_l2(ady, ady_ref))
    for i in range(6):
        assert rel_l2(grads[i], g_ref[i]) <= 1e-5, (NAMES[i], rel_l2(grads[i], g_ref[i]))


class _Requests:
    """phx_solve requests of one-problem solves of a 350 x 40 model at T = 3 on each engine, with the buffers they need."""

    def __init__(self, pb):
        import ctypes
        from phoenix_b200 import _lib
        self.lib, self.ctypes, self._lib = _lib.load(), ctypes, _lib
        G, H, T = self.G, self.H, self.T = 350, 40, 3
        net = make_net(pb, _weights(G, H, 91))
        self.packed, _, _, dev = pb.engine.packed_weights(net)
        self.ctx, self.sp = _lib.ctx(dev), pb.engine._stream_ptr(dev)
        self.y0 = torch.rand(2, 2, G, device="cuda")   # room for N = 2 problems of B = 2 rows
        self.yout = torch.empty(2, T, 2, G, device="cuda")
        self.gy = torch.rand(2, T, 2, G, device="cuda")
        self.adj = torch.empty(2, 2, G, device="cuda")
        self.flat = torch.empty(2, 4 * G * H + 2 * H + G, device="cuda")
        self.gparts = torch.empty(self.lib.phx_packed_grad_bytes(G, H) // 4, device="cuda")
        self.tarr = (ctypes.c_double * (2 * T))(0.0, 0.05, 0.1, 0.0, 0.05, 0.1)
        self.log = torch.zeros(16, 3, dtype=torch.float64).pin_memory()
        self.st = pb.engine._new_status_block(2)
        room = 16 + self.lib.phx_grid_workspace_bytes(1, T, 4)
        self.ws = {}
        for engine in ("resident", "rows", "stream"):
            size = {"resident": self.lib.phx_solve_workspace_bytes, "rows": self.lib.phx_rows_workspace_bytes,
                    "stream": self.lib.phx_stream_workspace_bytes}[engine]
            nb = max(size(self.ctx, G, H, 2, T, a) for a in (0, 1))   # B = 2 rows, or N = 2 rows problems
            self.ws[engine] = pb.engine._workspace(dev, nb + room, "solve" if engine != "stream" else "stream")

    def solve(self, which, adjoint, grid=(), method=2, **fields):
        """phx_solve of a one-problem, one-row rk4 solve on engine ``which`` (grid: the grid arrays in field order), with
        ``fields`` of the request overridden."""
        _lib = self._lib
        ws = self.ws[which]
        d = _lib.PhxSolveDesc(engine={"resident": 0, "rows": 1, "stream": 2}[which], adjoint=adjoint, G=self.G, H=self.H,
                              B=1, N=1, T=self.T, method=method, rtol=1e-7, atol=1e-9, max_num_steps=2 ** 31 - 1,
                              packed=self.packed.data_ptr(), t_host=self.ctypes.addressof(self.tarr),
                              workspace=ws.data_ptr(), workspace_bytes=ws.numel(), status=self.st.data_ptr())
        if adjoint:
            d.y_saved, d.grad_y, d.adj_y0 = self.yout.data_ptr(), self.gy.data_ptr(), self.adj.data_ptr()
            d.grads = (self.gparts if which == "rows" else self.flat).data_ptr()
            d.param_mask = _lib.PARAMS_ALL
        else:
            d.y0, d.y_out = self.y0.data_ptr(), self.yout.data_ptr()
        for name, x in zip(("grid_dt", "grid_steps", "grid_out_step", "grid_out_slope"), grid):
            setattr(d, name, x.data_ptr())
        for name, v in fields.items():
            setattr(d, name, v)
        return self.lib.phx_solve(self.ctx, self.ctypes.byref(d), self.sp)


@pytest.mark.gpu
def test_invalid_grids_are_refused_by_phx_solve(pb):
    """Every refusal of a step grid by phx_solve: PHX_ERR_INVALID before anything is enqueued -- a step count < 1, a
    negative or non-finite dt, an output step out of range or decreasing, a NaN slope, dopri5 -- for the resident, rows
    and streaming forward and adjoint solves; the valid grid next to them runs."""
    from phoenix_b200 import _lib
    rq = _Requests(pb)
    I32 = lambda *v: torch.tensor(v, dtype=torch.int32)   # noqa: E731
    F32 = lambda *v: torch.tensor(v, dtype=torch.float32)   # noqa: E731
    good_f = (F32(0.03, 0.02, 0.03, 0.02), I32(4), I32(1, 3), F32(-1.0, -1.0))
    good_a = (F32(0.03, 0.02, 0.03, 0.02), I32(2, 2))
    bad_f = [(F32(0.03), I32(0), I32(0, 0), F32(-1.0, -1.0)),                        # no steps
             (F32(0.03, -0.02, 0.03, 0.02), I32(4), I32(1, 3), F32(-1.0, -1.0)),   # negative dt
             (F32(0.03, float("inf"), 0.03, 0.02), I32(4), I32(1, 3), F32(-1.0, -1.0)),
             (F32(0.03, float("nan"), 0.03, 0.02), I32(4), I32(1, 3), F32(-1.0, -1.0)),
             (F32(0.03, 0.02, 0.03, 0.02), I32(4), I32(1, 4), F32(-1.0, -1.0)),    # output step out of range
             (F32(0.03, 0.02, 0.03, 0.02), I32(4), I32(-1, 3), F32(-1.0, -1.0)),
             (F32(0.03, 0.02, 0.03, 0.02), I32(4), I32(3, 1), F32(-1.0, -1.0)),    # decreasing output map
             (F32(0.03, 0.02, 0.03, 0.02), I32(4), I32(1, 3), F32(float("nan"), -1.0))]
    bad_a = [(F32(0.03, 0.02, 0.03), I32(2, 0)), (F32(0.03, -0.02, 0.03, 0.02), I32(2, 2)),
             (F32(0.03, float("inf"), 0.03, 0.02), I32(2, 2))]
    for engine in ("resident", "rows", "stream"):
        for g in bad_f:
            assert rq.solve(engine, 0, g) == -1, (engine, g)   # PHX_ERR_INVALID
        for g in bad_a:
            assert rq.solve(engine, 1, g) == -1, (engine, g)
        assert rq.solve(engine, 0, good_f, method=3) == -1 and rq.solve(engine, 1, good_a, method=3) == -1, engine  # dopri5
        assert rq.solve(engine, 0, good_f) == 0, (engine, _lib.last_error())
        torch.cuda.synchronize()
        assert rq.solve(engine, 1, good_a) == 0, (engine, _lib.last_error())
        torch.cuda.synchronize()


@pytest.mark.gpu
def test_phx_solve_refuses_the_combinations_no_engine_takes(pb):
    """phx_solve refuses, with PHX_ERR_INVALID and a message, what none of the engines takes: an unknown engine,
    `reversed` or forward-grid outputs on an adjoint solve, a param_mask on a forward solve, grid arrays without grid_dt,
    N != 1 on the streaming engine, B != 1 on the rows engine, `reversed` or a step log with N > 1 on the resident
    engine; the plain requests next to them run."""
    from phoenix_b200 import _lib
    rq = _Requests(pb)
    steps, out_step, slope = (torch.tensor(v, dtype=t) for v, t in
                              (((4,), torch.int32), ((1, 3), torch.int32), ((-1.0, -1.0), torch.float32)))
    refused = [("resident", 0, dict(engine=3)), ("stream", 1, dict(engine=-1)),
               ("resident", 1, dict(reversed=1)), ("rows", 1, dict(reversed=1)), ("stream", 1, dict(reversed=1)),
               ("resident", 0, dict(param_mask=_lib.PARAMS_ALL)), ("rows", 0, dict(param_mask=1)),
               ("stream", 0, dict(param_mask=_lib.NORM_SEMINORM)),
               ("resident", 1, dict(grid_out_step=out_step.data_ptr())), ("rows", 1, dict(grid_out_slope=slope.data_ptr())),
               ("resident", 0, dict(grid_steps=steps.data_ptr())), ("stream", 1, dict(grid_steps=steps.data_ptr())),
               ("stream", 0, dict(N=2)), ("stream", 1, dict(N=2)), ("rows", 0, dict(B=2)), ("rows", 1, dict(B=2)),
               ("resident", 0, dict(N=2, reversed=1)), ("resident", 0, dict(N=2, steplog=rq.log.data_ptr(), steplog_cap=16))]
    for engine, adjoint, fields in refused:
        assert rq.solve(engine, adjoint, **fields) == -1, (engine, adjoint, fields)
        assert _lib.last_error(), (engine, adjoint, fields)
    for engine, adjoint, fields in [("resident", 0, dict(reversed=1, steplog=rq.log.data_ptr(), steplog_cap=16)),
                                    ("resident", 0, dict(N=2, B=2)), ("resident", 1, dict(N=2, B=2)),
                                    ("rows", 0, dict(N=2)), ("stream", 0, dict(B=2, reversed=1))]:
        assert rq.solve(engine, adjoint, **fields) == 0, (engine, adjoint, fields, _lib.last_error())
        torch.cuda.synchronize()
