"""Gradients with respect to ``t`` in ``odeint_adjoint`` and ``odeint_adjoint_many`` (torchdiffeq 0.1.1 adjoint.py, backward
with ``t_requires_grad``).

The reference forms, before integrating output interval i = T-1 .. 1, ``dLd_i = func(t[i], y[i]) . grad_y[i]``, subtracts
it from the time cotangent ``vjp_t`` (the first entry of the augmented state), records it as ``time_vjps[i]`` and, after
the last interval, sets ``time_vjps[0] = vjp_t``.  ODENet is autonomous, so the solver carries vjp_t unchanged: the time
cotangents need no sweep.  vjp_t is still a block of dopri5's mixed norm, where it can set the backward's initial step.
The oracle module is pinned to the goldens, so its extension lives here: ``adjoint_backward_t`` takes the reference's
loop literally, with vjp_t carried through every interval's ``_solve``.  CPU tests pin the extension and the host logic;
GPU tests run every engine (resident, resident many, rows at 4 / 2 / 1 rows per pass, streaming)."""
import pytest
import torch

import phoenix_b200 as pbm
from phoenix_b200.torchdiffeq import _api
from oracle import phoenix_oracle as O
from golden_util import assert_logs_close, rel_l2
from test_gpu_adjoint_params import _oracle_problem
from test_gpu_adjoint_seminorm import ENGINES, _eid, _problem
from test_gpu_dopri5_options import solve_dopri5_x
from test_gpu_placements import make_net
from test_gpu_step_size import _Requests, solve_fixed_grid

NAMES = O.PARAM_ORDER


# ---- oracle extension (CPU) -----------------------------------------------------------------------------------------------
def adjoint_backward_t(w, t, y, grad_y, method="dopri5", rtol=1e-7, atol=1e-9, t_requires_grad=False, semi=False,
                       first_step=None, step_size=None, params=None, replay=None):
    """O.adjoint_backward with the augmented state's vjp_t carried from interval to interval, as the reference carries
    ``aug_state[0]``; with ``t_requires_grad`` it also forms the reference's time_vjps.  ``semi``: the seminorm (the
    norm of the first 1 + 2N entries); ``first_step`` (dopri5) starts every interval; ``step_size`` (fixed grids) steps
    every interval on its own grid.  ``params``: the adjoint set S as indices (None: all six) -- the default norm's
    parameter block holds only S (``adjoint_backward_s``), while all six cotangents are still integrated (the y / adj_y
    algebra never reads them); ``replay``: a dopri5 backward step log to take instead of the controller's steps
    (``O.Replay``; ``first_step`` is then only in the log).  Returns (adj_y0, [6 grads], StepLog, time_vjps in t's dtype
    or None)."""
    log = O.StepLog([])
    shape = y.shape[1:]
    N = y[0].numel()
    params_all = w.as_list()
    psz = [p.numel() for p in params_all]
    P = sum(psz)
    if semi:
        head = O.block_max_rms([1, N, N])
        norm = lambda x: head(x[:1 + 2 * N])   # noqa: E731
    elif params is None or sorted(set(params)) == list(range(6)):
        norm = O.block_max_rms([1, N, N, P])
    else:
        keep = torch.cat([torch.full((n,), i in set(params), dtype=torch.bool) for i, n in enumerate(psz)])
        ps = int(keep.sum())
        blocks = O.block_max_rms([1, N, N, ps] if ps else [1, N, N])
        norm = lambda x: blocks(torch.cat([x[:1 + 2 * N], x[1 + 2 * N:][keep]]))   # noqa: E731
    rp = None if replay is None else O.Replay(replay)

    def aug_reversed(tt, z):
        f, ybar, pbar = O.rhs_vjp(w, z[1:1 + N].reshape(shape), -z[1 + N:1 + 2 * N].reshape(shape))
        return -torch.cat([torch.zeros(1, dtype=z.dtype), f.reshape(-1), ybar.reshape(-1)]
                          + [p.reshape(-1) for p in pbar])

    def solve(z0, tt):
        if method != "dopri5":
            return solve_fixed_grid(aug_reversed, z0, tt, method, log, step_size)
        if first_step is None or rp is not None:
            return O._solve(aug_reversed, z0, tt, method, rtol, atol, norm, log, rp)
        return solve_dopri5_x(aug_reversed, z0, tt, rtol, atol, norm, log, first_step=first_step)

    with torch.no_grad():
        vjp_t = torch.zeros(1, dtype=y.dtype)
        time_vjps = torch.empty(len(t), dtype=t.dtype) if t_requires_grad else None
        adj_y = grad_y[-1].clone()
        adj_p = torch.zeros(P, dtype=y.dtype)
        cur_y = y[-1]
        for i in range(len(t) - 1, 0, -1):
            if t_requires_grad:
                d = O.rhs(w, y[i]).reshape(-1).dot(grad_y[i].reshape(-1))
                vjp_t = vjp_t - d
                time_vjps[i] = d
            z0 = torch.cat([vjp_t, cur_y.reshape(-1), adj_y.reshape(-1), adj_p])
            z = solve(z0, -t[i - 1:i + 1].flip(0))[1]
            vjp_t = z[:1]
            adj_p = z[1 + 2 * N:]
            cur_y = y[i - 1]
            adj_y = z[1 + N:1 + 2 * N].reshape(shape) + grad_y[i - 1]
        if rp is not None:
            rp.finish()
        if t_requires_grad:
            time_vjps[0] = vjp_t[0]
        grads, lo = [], 0
        for p, n in zip(params_all, psz):
            grads.append(adj_p[lo:lo + n].reshape(p.shape))
            lo += n
    return adj_y, grads, log, time_vjps


@pytest.mark.parametrize("method", ["dopri5", "rk4"])
def test_oracle_extension_without_t_grad_is_the_oracle(method):
    w, t, y, gy = _oracle_problem(method=method)
    a0, g0, l0 = O.adjoint_backward(w, t, y, gy, method=method)
    a1, g1, l1, tv = adjoint_backward_t(w, t, y, gy, method=method)
    assert tv is None
    assert torch.equal(a1, a0) and all(torch.equal(x, z) for x, z in zip(g1, g0))
    assert l1.steps == l0.steps and l1.nfe == l0.nfe


def _loss64(w, y0, t, target):
    y, _ = O.odeint(w, y0, t, method="dopri5", rtol=1e-10, atol=1e-12)
    return float(((y[1:] - target) ** 2).sum())


def test_oracle_time_vjps_match_finite_differences():
    """float64 oracle, dopri5 at rtol 1e-10, T = 3: time_vjps against central differences of the loss in each t_i."""
    w, _, y32, _ = _oracle_problem()
    wd = O.Weights(*[p.double() for p in w.as_list()])
    gen = torch.Generator().manual_seed(5)
    y0 = y32[0].double()
    target = torch.rand(2, *y0.shape, generator=gen, dtype=torch.float64)
    t = torch.tensor([0.0, 0.3, 0.6], dtype=torch.float64)
    y, _ = O.odeint(wd, y0, t, method="dopri5", rtol=1e-10, atol=1e-12)
    gy = torch.zeros_like(y)
    gy[1:] = 2.0 * (y[1:] - target)
    _, _, _, tv = adjoint_backward_t(wd, t, y, gy, rtol=1e-10, atol=1e-12, t_requires_grad=True)
    eps = 1e-4
    fd = []
    for i in range(3):
        e = torch.zeros(3, dtype=torch.float64)
        e[i] = eps
        fd.append((_loss64(wd, y0, t + e, target) - _loss64(wd, y0, t - e, target)) / (2 * eps))
    assert tv.dtype == torch.float64
    assert rel_l2(tv, torch.tensor(fd)) < 1e-5, (tv, fd)


def test_oracle_first_time_vjp_is_minus_the_sum_of_the_others():
    """time_vjps[0] = -sum(time_vjps[1:]) up to the rounding of the constant vjp_t in dopri5's dense output."""
    w, _, _, _ = _oracle_problem()
    gen = torch.Generator().manual_seed(6)
    y0 = torch.rand(1, w.G, generator=gen)
    t = torch.tensor([0.0, 0.2, 0.5, 0.6], dtype=torch.float64)
    y, _ = O.odeint(w, y0, t, method="dopri5")
    gy = 2.0 * (y - torch.rand(y.shape, generator=gen))
    gy[0] = 0
    _, _, _, tv = adjoint_backward_t(w, t, y, gy, t_requires_grad=True)
    s = float(tv[1:].sum())
    assert abs(float(tv[0]) + s) <= 1e-5 * float(tv[1:].abs().sum()), (tv, s)


# ---- host logic (CPU) ------------------------------------------------------------------------------------------------------
def _cpu_net():
    torch.manual_seed(0)
    return pbm.ODENet("cpu", 12, neurons=4)


class _Ctx:
    """Stands in for an autograd context."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


@pytest.mark.parametrize("many", [False, True])
def test_odeint_refuses_t_grad_and_decreasing_t_stays_refused(many):
    net = _cpu_net()
    y0 = torch.rand(1, 12)
    t = torch.tensor([0.0, 1.0], requires_grad=True)
    with pytest.raises(NotImplementedError, match="odeint_adjoint"):
        pbm.odeint(net, y0, t)
    td = torch.tensor([1.0, 0.0], requires_grad=True)
    if many:
        with pytest.raises(AssertionError, match="increasing"):
            pbm.odeint_adjoint_many(net, y0.unsqueeze(0), td.unsqueeze(0))
    else:
        with pytest.raises(NotImplementedError, match="decreasing"):
            pbm.odeint_adjoint(net, y0, td)


@pytest.mark.parametrize("many", [False, True])
def test_apply_gets_t_only_when_it_needs_a_gradient(monkeypatch, many):
    got = []
    cls = _api.OdeintAdjointManyMethod if many else _api.OdeintAdjointMethod
    monkeypatch.setattr(cls, "apply", lambda *args: got.append(args))
    net = _cpu_net()
    y0 = torch.rand(1, 12)
    for rg in (False, True):
        t = torch.tensor([0.0, 1.0], dtype=torch.float64, requires_grad=rg)
        if many:
            pbm.odeint_adjoint_many(net, y0.unsqueeze(0), t.unsqueeze(0))
        else:
            pbm.odeint_adjoint(net, y0, t)
    assert len(got[0]) == 15 and all(torch.is_tensor(a) for a in got[0][8:])
    assert len(got[1]) == 16 and got[1][:8] == got[0][:8] and got[1][15].requires_grad
    with torch.no_grad():   # no graph: t is not an input
        t = torch.tensor([0.0, 1.0], requires_grad=True)
        if many:
            pbm.odeint_adjoint_many(net, y0.unsqueeze(0), t.unsqueeze(0))
        else:
            pbm.odeint_adjoint(net, y0, t)
    assert len(got[2]) == 15


@pytest.mark.parametrize("many", [False, True])
def test_backward_without_t_grad_is_unchanged(monkeypatch, many):
    calls = []

    def fake(*a, **k):
        calls.append(k)
        return torch.zeros(1, 12), [torch.ones(1) * i for i in range(6)]

    monkeypatch.setattr(_api.engine, "solve_adjoint", fake)
    monkeypatch.setattr(_api.engine, "solve_adjoint_many", fake)
    monkeypatch.setattr(_api.engine, "time_vjp", lambda *a: pytest.fail("time_vjp without t grad"))
    ctx = _Ctx(saved_tensors=(torch.zeros(2, 1, 12),), adj=("dopri5", 1e-7, 1e-9, 100, 0x3F, None),
               needs_input_grad=(False,) * 9 + (True,) * 6, group=None, func=_cpu_net(), tl=[0.0, 1.0],
               t_rows=[[0.0, 1.0]], t_is_f32=True)
    cls = _api.OdeintAdjointManyMethod if many else _api.OdeintAdjointMethod
    out = cls.backward(ctx, torch.zeros(2, 1, 12))
    assert len(out) == 15 and out[:9] == (None,) * 9 and all(torch.is_tensor(g) for g in out[9:])
    assert calls == [{}]


def test_group_key_separates_t_grad():
    saved = _api.DEFER_ADJOINT
    _api.DEFER_ADJOINT = True
    try:
        net = _cpu_net()
        y0 = torch.rand(1, 12)
        keys = []
        for flags in ((False,) * 9 + (True,) * 6, (False,) * 9 + (True,) * 6 + (True,)):
            ctx = _Ctx(needs_input_grad=flags)
            _api._register_node(ctx, net, y0, [0.0, 1.0], True, ("dopri5", 1e-7, 1e-9, 100, 0x3F, None))
            keys.append(ctx.group)
        assert keys[0] is not None and keys[1] is not None and keys[0] != keys[1]
    finally:
        _api.DEFER_ADJOINT = saved


@pytest.mark.parametrize("many", [False, True])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_t_only_backward_runs_no_sweep(monkeypatch, many, dtype):
    def boom(*a, **k):
        raise AssertionError("a sweep ran")

    monkeypatch.setattr(_api.engine, "solve_adjoint", boom)
    monkeypatch.setattr(_api.engine, "solve_adjoint_many", boom)
    T = 3
    n = 2 if many else 1
    tg = torch.arange(n * T, dtype=torch.float32).reshape(n, T) + 0.5
    monkeypatch.setattr(_api.engine, "time_vjp", lambda net, y, gy: (tg, torch.zeros(n, T - 1)))
    ctx = _Ctx(saved_tensors=(torch.zeros(n, T, 1, 12) if many else torch.zeros(T, 1, 12),),
               adj=("dopri5", 1e-7, 1e-9, 100, 0x0, None), needs_input_grad=(False,) * 15 + (True,), group=None,
               func=_cpu_net(), tl=[0.0, 1.0, 2.0], t_rows=[[0.0, 1.0, 2.0]] * n, t_is_f32=dtype == torch.float32,
               t_meta=(dtype, torch.device("cpu")))
    cls = _api.OdeintAdjointManyMethod if many else _api.OdeintAdjointMethod
    out = cls.backward(ctx, torch.zeros_like(ctx.saved_tensors[0]))
    assert len(out) == 16 and out[:15] == (None,) * 15
    assert out[15].dtype == dtype and out[15].device.type == "cpu"
    assert torch.equal(out[15], (tg if many else tg[0]).to(dtype))


# ---- GPU -----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pb():
    pbm.set_sync_errors(True)
    yield pbm
    pbm.set_step_logging(False)
    pbm.engine.FORCE_ENGINE = None


# (name, method, adjoint_options, oracle keywords)
VARIANTS = [("dopri5", "dopri5", None, {}), ("seminorm", "dopri5", {"norm": "seminorm"}, {"semi": True}),
            ("first_step", "dopri5", {"first_step": 0.02}, {"first_step": 0.02}),
            ("rk4-step", "rk4", {"step_size": 0.03}, {"step_size": 0.03})]


def _run(pb, net, y0, t, loss, method, engine, many, adjoint_options=None, logging=True, rtol=1e-5, atol=1e-7):
    """Forward + backward on the GPU with a t that requires grad (a copy of ``t``).  ``loss(y)`` is the loss of the
    outputs.  Returns y, adj_y0, the six .grad, t.grad and the backward step logs (None when not logged)."""
    saved = pb.engine.FORCE_ENGINE
    pb.engine.FORCE_ENGINE = engine
    pb.set_step_logging(logging)
    plist = list(net.parameters())
    try:
        net.zero_grad(set_to_none=True)
        y0g = y0.cuda().requires_grad_(True)
        tg = t.clone().requires_grad_(True)
        solve = pb.odeint_adjoint_many if many else pb.odeint_adjoint
        y = solve(net, y0g, tg, rtol=rtol, atol=atol, method=method, adjoint_options=adjoint_options)
        loss(y).backward()
        logs = None
        if logging:
            logs = [pb.last_step_log(i) for i in range(y0.shape[0])] if many else [pb.last_step_log()]
        return (y.detach().cpu(), y0g.grad.cpu(), [p.grad.detach().cpu().clone() for p in plist], tg.grad, logs)
    finally:
        pb.set_step_logging(False)
        pb.engine.FORCE_ENGINE = saved


def _oracle(w, y0, t, gys, many, method, rtol, atol, with_logs0=False, **kw):
    """fp32 oracle with t grad: y, adj_y0, the gradients summed over the problems, t.grad and the backward step logs;
    with ``with_logs0`` also the backward logs of the same problems without t grad.  ``gys(i, y)``: the loss cotangent
    of problem i's outputs y."""
    probs = [(y0[i], t[i]) for i in range(y0.shape[0])] if many else [(y0, t)]
    ys, adys, gsum, tvs, logs, logs0 = [], [], None, [], [], []
    for k, (y0i, ti) in enumerate(probs):
        yr, _ = O.odeint(w, y0i, ti, method=method, rtol=rtol, atol=atol)
        gy = gys(k, yr)
        ar, gr, blog, tv = adjoint_backward_t(w, ti, yr, gy, method, rtol, atol, t_requires_grad=True, **kw)
        if with_logs0:
            logs0.append(adjoint_backward_t(w, ti, yr, gy, method, rtol, atol, **kw)[2].steps)
        ys.append(yr)
        adys.append(ar)
        tvs.append(tv)
        gsum = gr if gsum is None else [a + b for a, b in zip(gsum, gr)]
        logs.append(blog.steps)
    st = (lambda v: torch.stack(v)) if many else (lambda v: v[0])
    return st(ys), st(adys), gsum, st(tvs), logs, logs0


def _sq_loss(target, many):
    """The loss sum((y[1:] - target)^2) on the GPU and its cotangent for the oracle's problem k."""
    def gys(k, yr):
        gy = torch.zeros_like(yr)
        gy[1:] = 2.0 * (yr[1:] - (target[k] if many else target))
        return gy
    return (lambda y: (((y[:, 1:] if many else y[1:]) - target.cuda()) ** 2).sum()), gys


@pytest.mark.gpu
@pytest.mark.parametrize("variant", VARIANTS, ids=[v[0] for v in VARIANTS])
@pytest.mark.parametrize("e", ENGINES, ids=[_eid(e) for e in ENGINES])
def test_t_grad_against_oracle(pb, e, variant):
    """t.grad (rel-L2 <= 1e-5), y, adj_y0 and the gradients (the tolerances of test_dopri5_seminorm_against_oracle)
    against the oracle extension, for T = 2 and 4 and a float32 and a float64 t; dopri5 backward logs to the oracle's."""
    engine, G, H, shape, many, _ = e
    name, method, aopts, okw = variant
    rtol, atol = 1e-5, 1e-7
    logging = method == "dopri5" and not (engine == "resident" and many)
    for T in (2, 4):
        w, y0, t, target = _problem(G, H, shape, many, tuple(0.1 * k for k in range(T)), 11)
        net = make_net(pb, w)
        for dtype in (torch.float32, torch.float64):
            tt = t.to(dtype)
            what = (_eid(e), name, T, str(dtype))
            loss, gys = _sq_loss(target, many)
            y, ady, grads, tgrad, logs = _run(pb, net, y0, tt, loss, method, engine, many, aopts, logging, rtol, atol)
            y_r, ady_r, g_r, tv_r, logs_r, _ = _oracle(w, y0, tt, gys, many, method, rtol, atol, **okw)
            assert tgrad.shape == tt.shape and tgrad.dtype == dtype and tgrad.device == tt.device, what
            assert rel_l2(tgrad, tv_r) <= 1e-5, (what, tgrad, tv_r)
            assert rel_l2(y, y_r) < 1e-5, what
            assert rel_l2(ady, ady_r) < 1e-5, (what, rel_l2(ady, ady_r))
            for i in range(6):
                assert rel_l2(grads[i], g_r[i]) < 5e-5, (what, NAMES[i], rel_l2(grads[i], g_r[i]))
            if logs is not None:
                for i, (mine, r) in enumerate(zip(logs, logs_r)):
                    assert_logs_close(mine, r, 0.25, "%s bwd %d" % (what, i))


CONSTRUCTED = [("resident", (1, 350), False), ("resident", (3, 1, 350), True), ("rows", (3, 1, 350), True),
               ("stream", (2, 350), False)]


@pytest.mark.gpu
@pytest.mark.parametrize("engine,shape,many", CONSTRUCTED, ids=["%s-%s" % (c[0], "x".join(map(str, c[1])))
                                                                for c in CONSTRUCTED])
def test_time_block_decides_the_first_backward_dt(pb, engine, shape, many):
    """G = 350, y0 ~ 1e-4 and grad_y = 1e-4 sign(f(y(t1))), rtol 1e-5, atol 1e-7: y and adj_y are so small that vjp_t is
    the largest block of d0 in Hairer's estimate, and the backward's first dt is not the one of a t without grad.  The
    kernels' backward logs follow the oracle's (first dt to 1e-4)."""
    rtol, atol = 1e-5, 1e-7
    w = O.make_weights(350, 40, 31, dense=True, neg_mult_frac=0.2)
    gen = torch.Generator().manual_seed(32)
    y0 = 1e-4 * torch.rand(*shape, generator=gen)
    times = torch.tensor([0.0, 0.01], dtype=torch.float64)
    t = times.expand(shape[0], 2).contiguous() if many else times
    # the loss (y(t1) . c) with c = 1e-4 sign(f(y(t1))) of the oracle's solve
    cs = []
    for k in range(shape[0] if many else 1):
        yr, _ = O.odeint(w, y0[k] if many else y0, times, method="dopri5", rtol=rtol, atol=atol)
        cs.append(1e-4 * torch.sign(O.rhs(w, yr[1])))
    c = torch.stack(cs) if many else cs[0]

    def gys(k, yr):
        gy = torch.zeros_like(yr)
        gy[1] = c[k] if many else c
        return gy

    _, _, _, _, logs_r, logs0 = _oracle(w, y0, t, gys, many, "dopri5", rtol, atol, with_logs0=True)
    for mine, r in zip(logs0, logs_r):
        assert abs(mine[0][1] - r[0][1]) > 1e-3 * r[0][1], (mine[0], r[0])
    net = make_net(pb, w)
    loss = lambda y: ((y[:, 1] if many else y[1]) * c.cuda()).sum()   # noqa: E731
    _, _, _, _, logs = _run(pb, net, y0, t, loss, "dopri5", engine, many, None, engine != "resident" or not many,
                            rtol, atol)
    if logs is not None:
        for i, (mine, r) in enumerate(zip(logs, logs_r)):
            assert_logs_close(mine, r, 0.25, "%s bwd %d" % (engine, i), first_rtol=1e-4)


@pytest.mark.gpu
def test_per_sample_loop_with_t_grad_matches_many(pb):
    """The literal loop of training_step with t requiring grad: every deferred node computes its own time cotangents and
    the last one runs the lock-step sweep with all of their t_vjp rows.  t.grad equals odeint_adjoint_many's to 1e-6,
    the parameter gradients as test_odeint_adjoint_many_equals_the_per_sample_loop requires (1e-6)."""
    G, H, N = 690, 40, 6
    w = O.make_weights(G, H, 21, dense=True, neg_mult_frac=0.2)
    gen = torch.Generator().manual_seed(22)
    y0 = torch.rand(N, 1, G, generator=gen)
    t = torch.rand(N, 1, generator=gen, dtype=torch.float64) + torch.tensor([0.0, 0.1], dtype=torch.float64)
    target = torch.rand(N, 1, G, generator=gen)
    net = make_net(pb, w)
    params = list(net.parameters())
    for method in ("rk4", "dopri5"):
        net.zero_grad(set_to_none=True)
        tl = t.clone().requires_grad_(True)
        preds = [pb.odeint_adjoint(net, y0[i].cuda(), tl[i], method=method)[1] for i in range(N)]
        torch.mean((torch.stack(preds) - target.cuda()) ** 2).backward()
        loop = [p.grad.clone() for p in params]
        net.zero_grad(set_to_none=True)
        tm = t.clone().requires_grad_(True)
        y = pb.odeint_adjoint_many(net, y0.cuda(), tm, method=method)
        torch.mean((y[:, 1] - target.cuda()) ** 2).backward()
        assert tl.grad.shape == (N, 2) and tm.grad.shape == (N, 2)
        assert rel_l2(tl.grad, tm.grad) < 1e-6, (method, tl.grad, tm.grad)
        for i in range(6):
            assert rel_l2(loop[i].cpu(), params[i].grad.cpu()) < 1e-6, (method, NAMES[i])


@pytest.mark.gpu
def test_directional_derivative_in_t(pb):
    """(L(t + eps e1) - L(t - eps e1)) / 2 eps of the GPU solve, float64 t, against t.grad[1] (rel. 1e-3), and a zero
    gradient for a single output time."""
    w, y0, t, target = _problem(350, 40, (1, 350), False, (0.0, 0.5, 1.0), 61)
    net = make_net(pb, w)
    loss = lambda y: ((y[1:] - target.cuda()) ** 2).sum()   # noqa: E731
    tg = _run(pb, net, y0, t, loss, "dopri5", "resident", False, None, False, 1e-7, 1e-9)[3]
    eps = 1e-3
    e = torch.tensor([0.0, eps, 0.0], dtype=torch.float64)
    with torch.no_grad():
        lp = float(loss(pb.odeint(net, y0.cuda(), t + e, rtol=1e-7, atol=1e-9)))
        lm = float(loss(pb.odeint(net, y0.cuda(), t - e, rtol=1e-7, atol=1e-9)))
    fd = (lp - lm) / (2 * eps)
    assert abs(fd - float(tg[1])) <= 1e-3 * abs(float(tg[1])), (fd, tg)
    t1 = torch.tensor([0.5], dtype=torch.float64, requires_grad=True)
    y0g = y0.cuda().requires_grad_(True)
    pb.odeint_adjoint(net, y0g, t1).sum().backward()
    assert torch.equal(t1.grad, torch.zeros(1, dtype=torch.float64))


@pytest.mark.gpu
def test_phx_solve_takes_t_vjp_on_adjoint_solves_only(pb):
    """t_vjp on a forward request: PHX_ERR_INVALID on every engine.  On a fixed-grid adjoint request it is accepted and
    changes nothing; on a dopri5 one a NaN time cotangent is the non-finite state of the reference's assertion."""
    from phoenix_b200 import _lib
    rq = _Requests(pb)
    tv = torch.zeros(1, rq.T - 1, device="cuda")
    nan = torch.full((1, rq.T - 1), float("nan"), device="cuda")
    for engine in ("resident", "rows", "stream"):
        assert rq.solve(engine, 0, t_vjp=tv.data_ptr()) == -1, engine
        assert "t_vjp" in _lib.last_error(), engine
        assert rq.solve(engine, 0) == 0, (engine, _lib.last_error())   # the saved outputs of the adjoint requests
        torch.cuda.synchronize()
        out = []
        for ptr in (None, tv.data_ptr()):
            assert rq.solve(engine, 1, t_vjp=ptr) == 0, (engine, _lib.last_error())
            torch.cuda.synchronize()
            out.append((rq.adj.clone(), (rq.gparts if engine == "rows" else rq.flat).clone()))
        assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1]), engine
        assert rq.solve(engine, 1, method=3, t_vjp=nan.data_ptr()) == 0, (engine, _lib.last_error())
        torch.cuda.synchronize()
        assert pb.engine._status_struct(rq.st[0]).code == _lib.ST_NONFINITE, engine
