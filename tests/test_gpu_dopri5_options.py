"""The dopri5 step-control options ``first_step``, ``safety``, ``ifactor`` and ``dfactor`` (torchdiffeq 0.1.1
rk_common.py:111-228, misc.py:94-103), forward and adjoint.

``first_step`` replaces Hairer's initial-step estimate (misc.py:47-86): f0 is still evaluated, the second evaluation and
the norms are not, and the first attempted dt is ``first_step`` -- of every output interval in the backward, which
integrates each interval with its own ``odeint`` call.  ``safety``, ``ifactor`` and ``dfactor`` are the constants of the
step-size controller.  The oracle module is pinned to the goldens, so its extension lives here: copies of
``_solve_dopri5`` and ``adjoint_backward`` that take the four options.  CPU tests pin the extension and the host logic;
GPU tests run every engine (resident, resident many, rows at 4 / 2 / 1 rows per pass, streaming)."""
import math

import pytest
import torch

import phoenix_b200 as pbm
from phoenix_b200.torchdiffeq import _api
from oracle import phoenix_oracle as O
from golden_util import assert_logs_close, rel_l2
from test_gpu_adjoint_params import _oracle_problem
from test_gpu_adjoint_seminorm import ENGINES, _eid, _problem
from test_gpu_placements import make_net
from test_gpu_step_size import _Requests

NAMES = O.PARAM_ORDER
DEFAULTS = dict(safety=0.9, ifactor=10.0, dfactor=0.2)


# ---- oracle extension (CPU) -----------------------------------------------------------------------------------------------
def next_dt_x(dt, ratio, safety=0.9, ifactor=10.0, dfactor=0.2):
    """O._next_dt with the controller constants as arguments (misc.py:94-103, order 5)."""
    if ratio == 0:
        return dt * ifactor
    dfactor = 1.0 if ratio < 1 else dfactor
    r = ratio.to(dt.dtype)
    factor = min(ifactor, max(safety / float(r ** torch.tensor(0.2, dtype=dt.dtype)), dfactor))
    if math.isnan(float(r)):
        factor = float("nan")
    return dt * factor


def solve_dopri5_x(func, y0, t, rtol, atol, norm, log, first_step=None, safety=0.9, ifactor=10.0, dfactor=0.2):
    """O._solve_dopri5 with the four options: ``first_step`` (float64) replaces Hairer's estimate and its second
    evaluation; the controller takes the three constants."""
    dtype = y0.dtype
    t = t.to(torch.float64)
    rt = torch.as_tensor(rtol, dtype=torch.float64)
    at = torch.as_tensor(atol, dtype=torch.float64)
    beta = [torch.tensor(b, dtype=torch.float64).to(dtype) for b in O.DP_BETA]
    c_err = torch.tensor(O.DP_C_ERROR, dtype=torch.float64).to(dtype)
    c_mid = torch.tensor(O.DP_C_MID, dtype=torch.float64).to(dtype)

    def f(tt, yy):
        log.nfe += 1
        return func(tt.to(dtype), yy)

    out = torch.empty(len(t), *y0.shape, dtype=dtype)
    out[0] = y0
    f0 = f(t[0], y0)
    if first_step is None:
        dt = O._initial_step(f, t[0], y0, f0, rt, at, norm)
    else:
        dt = torch.tensor(float(first_step), dtype=torch.float64)
    y, t0, t1 = y0, t[0], t[0]
    coeff = [y0] * 5
    for i in range(1, len(t)):
        n = 0
        while t[i] > t1:
            assert t1 + dt > t1, "underflow in dt {}".format(dt.item())
            assert torch.isfinite(y).all(), "non-finite values in state `y`: {}".format(y)
            ts, dts = t1.to(dtype), dt.to(dtype)
            k = torch.empty(*f0.shape, 7, dtype=dtype)
            k[..., 0] = f0
            for s_idx in range(6):
                yi = y + k[..., :s_idx + 1].matmul(beta[s_idx] * dts).view_as(f0)
                k[..., s_idx + 1] = f(ts + O.DP_ALPHA[s_idx] * dts, yi)
            y1, f1 = yi, k[..., 6]
            err = k.matmul(dts * c_err)
            tol = at + rt * torch.max(y.abs(), y1.abs())
            ratio = norm(err / tol)
            accept = bool(ratio <= 1)
            log.steps.append((float(t1), float(dt), accept))
            if accept:
                ymid = y + k.matmul(dts * c_mid).view_as(y)
                ka, kb = k[..., 0], k[..., 6]
                coeff = [y, dts * ka,
                         dts * (kb - 4 * ka) - 11 * y - 5 * y1 + 16 * ymid,
                         dts * (5 * ka - 3 * kb) + 18 * y + 14 * y1 - 32 * ymid,
                         2 * dts * (kb - ka) - 8 * (y1 + y) + 16 * ymid]
                t0, t1 = t1, t1 + dt
                y, f0 = y1, f1
            else:
                t0 = t1
            dt = next_dt_x(dt, ratio, safety, ifactor, dfactor)
            n += 1
        assert (t0 <= t[i]) & (t[i] <= t1), "invalid interpolation"
        x = (t[i] - t0) / (t1 - t0)
        total = coeff[0] + x * coeff[1]
        xp = x
        for c in coeff[2:]:
            xp = xp * x
            total = total + xp * c
        out[i] = total
    return out


def odeint_x(w, y0, t, rtol=1e-7, atol=1e-9, **opts):
    """O.odeint (dopri5, increasing t) with the options."""
    log = O.StepLog([])
    with torch.no_grad():
        y = solve_dopri5_x(lambda tt, yy: O.rhs(w, yy), y0, t, rtol, atol, O.rms, log, **opts)
    return y, log


def adjoint_backward_x(w, t, y, grad_y, rtol=1e-7, atol=1e-9, **opts):
    """O.adjoint_backward (dopri5) with the options; ``first_step`` starts every output interval."""
    log = O.StepLog([])
    shape = y.shape[1:]
    N = y[0].numel()
    params = w.as_list()
    psz = [p.numel() for p in params]
    P = sum(psz)
    norm = O.block_max_rms([1, N, N, P])

    def aug_reversed(tt, z):
        f, ybar, pbar = O.rhs_vjp(w, z[1:1 + N].reshape(shape), -z[1 + N:1 + 2 * N].reshape(shape))
        return -torch.cat([torch.zeros(1, dtype=z.dtype), f.reshape(-1), ybar.reshape(-1)]
                          + [p.reshape(-1) for p in pbar])

    with torch.no_grad():
        adj_y = grad_y[-1].clone()
        adj_p = torch.zeros(P, dtype=y.dtype)
        cur_y = y[-1]
        for i in range(len(t) - 1, 0, -1):
            z0 = torch.cat([torch.zeros(1, dtype=y.dtype), cur_y.reshape(-1), adj_y.reshape(-1), adj_p])
            z = solve_dopri5_x(aug_reversed, z0, -t[i - 1:i + 1].flip(0), rtol, atol, norm, log, **opts)[1]
            adj_p = z[1 + 2 * N:]
            cur_y = y[i - 1]
            adj_y = z[1 + N:1 + 2 * N].reshape(shape) + grad_y[i - 1]
        grads, lo = [], 0
        for p, n in zip(params, psz):
            grads.append(adj_p[lo:lo + n].reshape(p.shape))
            lo += n
    return adj_y, grads, log


def interval_starts(log, t):
    """The first attempt of every backward interval: the first logged step at t0 == -t[i], from the last interval."""
    out = []
    for i in range(len(t) - 1, 0, -1):
        out.append(next(s for s in log if s[0] == -float(t[i])))
    return out


@pytest.mark.parametrize("opts", [{}, DEFAULTS], ids=["none", "explicit-defaults"])
def test_oracle_extension_equals_the_oracle(opts):
    w, t, y, gy = _oracle_problem()
    y0 = y[0]
    yr, lr = O.odeint(w, y0, t, method="dopri5")
    yx, lx = odeint_x(w, y0, t, **opts)
    assert torch.equal(yx, yr) and lx.steps == lr.steps and lx.nfe == lr.nfe
    ar, gr, br = O.adjoint_backward(w, t, yr, gy, method="dopri5")
    ax, gx, bx = adjoint_backward_x(w, t, yr, gy, **opts)
    assert torch.equal(ax, ar) and all(torch.equal(a, b) for a, b in zip(gx, gr))
    assert bx.steps == br.steps and bx.nfe == br.nfe


def test_oracle_first_step_starts_every_solve():
    w, t, y, gy = _oracle_problem()
    h = 0.0123
    yx, lx = odeint_x(w, y[0], t, first_step=h)
    assert lx.steps[0][1] == h and lx.nfe == 1 + 6 * len(lx.steps)
    _, _, bx = adjoint_backward_x(w, t, yx, gy, first_step=h)
    starts = interval_starts(bx.steps, t)
    assert [s[1] for s in starts] == [h] * (len(t) - 1)
    assert bx.nfe == (len(t) - 1) + 6 * len(bx.steps)
    # Hairer's estimate passed back as first_step changes nothing but the count
    _, l0 = odeint_x(w, y[0], t)
    y1, l1 = odeint_x(w, y[0], t, first_step=l0.steps[0][1])
    assert l1.steps == l0.steps and l1.nfe == l0.nfe - 1


def test_controller_hand_check():
    dt = torch.tensor(0.25, dtype=torch.float64)
    c = dict(safety=0.8, ifactor=5.0, dfactor=0.5)
    r = lambda v: torch.tensor(v, dtype=torch.float32)   # noqa: E731
    assert float(next_dt_x(dt, r(0.0), **c)) == 0.25 * 5.0
    # ratio < 1: dfactor becomes 1, so an accepted step never shrinks, and it grows by safety / ratio^(1/5) up to ifactor
    assert float(next_dt_x(dt, r(0.5), **c)) == 0.25
    assert float(next_dt_x(dt, r(0.01), **c)) == 0.25 * (0.8 / float(torch.tensor(0.01, dtype=torch.float32).double()
                                                                        ** 0.2))
    assert float(next_dt_x(dt, r(1e-12), **c)) == 0.25 * 5.0
    # ratio > 1: safety / ratio^(1/5) is floored at dfactor
    assert float(next_dt_x(dt, r(100.0), **c)) == 0.25 * 0.5
    assert float(next_dt_x(dt, r(2.0), **c)) == 0.25 * (0.8 / 2.0 ** 0.2)
    assert math.isnan(float(next_dt_x(dt, r(float("nan")), **c)))


# ---- host logic (CPU) -------------------------------------------------------------------------------------------------------
def _cpu_net():
    torch.manual_seed(0)
    return pbm.ODENet("cpu", 12, neurons=4)


def _captured(monkeypatch, many, **kw):
    """The (fwd, adj) tuples an entry point hands its autograd node."""
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
        pbm.odeint_adjoint_many(net, y0.unsqueeze(0), t.unsqueeze(0), **kw)
    else:
        pbm.odeint_adjoint(net, y0, t, **kw)
    return got["fwd"], got["adj"]


def test_engine_keyword_only_with_options(monkeypatch):
    calls = []
    monkeypatch.setattr(_api.engine, "solve_forward", lambda *a, **k: calls.append(k))
    net = _cpu_net()
    y0 = torch.rand(1, 12)
    t = torch.tensor([0.0, 1.0])
    with torch.no_grad():
        pbm.odeint(net, y0, t)
        pbm.odeint(net, y0, t, options=dict(max_num_steps=50))
        pbm.odeint(net, y0, t, options=dict(first_step=0.5))
        pbm.odeint(net, y0, t, method="dopri5",
                   options=dict(safety=torch.tensor(0.8, dtype=torch.float64), dfactor=0.3))
    assert calls == [{}, {}, {"step_control": (0.5, 0.0, 0.0, 0.0)}, {"step_control": (0.0, 0.8, 0.0, 0.3)}]


@pytest.mark.parametrize("many", [False, True])
def test_adjoint_options_inherit_and_override(monkeypatch, many):
    # without options the tuples are what they always were
    fwd, adj = _captured(monkeypatch, many)
    assert len(fwd) == 2 and len(adj) == 6
    fwd, adj = _captured(monkeypatch, many, options=dict(first_step=0.5, ifactor=4))
    assert fwd[2] == (0.5, 0.0, 4.0, 0.0) and adj[6] == (0.5, 0.0, 4.0, 0.0)
    fwd, adj = _captured(monkeypatch, many, options=dict(first_step=0.5), adjoint_options=dict(safety=0.7))
    assert fwd[2] == (0.5, 0.0, 0.0, 0.0) and adj[6] == (0.0, 0.7, 0.0, 0.0)
    fwd, adj = _captured(monkeypatch, many, options=dict(first_step=0.5), adjoint_options=dict(max_num_steps=9))
    assert len(adj) == 6 and adj[3] == 9
    fwd, adj = _captured(monkeypatch, many, adjoint_options=dict(first_step=0.25, norm="seminorm"))
    assert len(fwd) == 2 and adj[6] == (0.25, 0.0, 0.0, 0.0) and adj[4] == 0x7F


class _Ctx:
    def __init__(self, **kw):
        self.__dict__.update(kw)


@pytest.mark.parametrize("many", [False, True])
def test_backward_passes_the_step_control(monkeypatch, many):
    calls = []

    def fake(*a, **k):
        calls.append(k)
        return torch.zeros(1, 12), [torch.zeros(1)] * 6

    monkeypatch.setattr(_api.engine, "solve_adjoint_many" if many else "solve_adjoint", fake)
    cls = _api.OdeintAdjointManyMethod if many else _api.OdeintAdjointMethod
    for ctl in (None, (0.5, 0.0, 0.0, 0.0)):
        adj = _api._with_control(("dopri5", 1e-7, 1e-9, 100, 0x3F, None), ctl)
        ctx = _Ctx(saved_tensors=(torch.zeros(2, 1, 12),), adj=adj,
                   needs_input_grad=(False,) * 9 + (True,) * 6, group=None, func=_cpu_net(), tl=[0.0, 1.0],
                   t_rows=[[0.0, 1.0]], t_is_f32=True)
        cls.backward(ctx, torch.zeros(2, 1, 12))
    assert calls == [{}, {"step_control": (0.5, 0.0, 0.0, 0.0)}]


def test_deferred_group_key_includes_the_step_control(monkeypatch):
    monkeypatch.setattr(_api, "DEFER_ADJOINT", True)
    net = _cpu_net()
    y0 = torch.rand(1, 12)
    keys = []
    for ctl in (None, (0.5, 0.0, 0.0, 0.0), (0.25, 0.0, 0.0, 0.0), (0.0, 0.8, 0.0, 0.0)):
        ctx = _Ctx(needs_input_grad=(False,) * 9 + (True,) * 6)
        _api._register_node(ctx, net, y0, [0.0, 1.0], True,
                            _api._with_control(("dopri5", 1e-7, 1e-9, 100, 0x3F, None), ctl))
        keys.append(ctx.group)
    assert None not in keys and len(set(keys)) == 4


@pytest.mark.parametrize("many", [False, True])
def test_refusals(monkeypatch, many):
    monkeypatch.setattr(_api.OdeintAdjointMethod, "apply", lambda *a: None)
    monkeypatch.setattr(_api.OdeintAdjointManyMethod, "apply", lambda *a: None)
    net = _cpu_net()
    y0 = torch.rand(1, 12)
    t = torch.tensor([0.0, 1.0])
    solve = (lambda **kw: pbm.odeint_adjoint_many(net, y0.unsqueeze(0), t.unsqueeze(0), **kw)) if many else \
        (lambda **kw: pbm.odeint_adjoint(net, y0, t, **kw))
    for key in ("first_step", "safety", "ifactor", "dfactor"):
        for method in ("euler", "midpoint", "rk4"):
            with pytest.raises(NotImplementedError, match=key):
                solve(method=method, options={key: 0.1})
        for bad in (0, 0.0, -1.0, float("inf"), float("nan"), torch.tensor(-0.5)):
            with pytest.raises(ValueError, match=key):
                solve(options={key: bad})
            with pytest.raises(ValueError, match=key):
                solve(adjoint_options={key: bad})
        with pytest.raises(NotImplementedError, match="0-dimensional"):
            solve(options={key: torch.tensor([0.1])})
        solve(options={key: torch.tensor(0.1)})
    if not many:
        # a fixed-grid backward inherits the forward's dopri5 options: refused like step_size with dopri5
        with pytest.raises(NotImplementedError, match="first_step"):
            solve(method="dopri5", options=dict(first_step=0.1), adjoint_method="rk4")
    for key in ("grid_points", "eps"):
        with pytest.raises(NotImplementedError, match=key):
            solve(options={key: 0.1, "first_step": 0.1})


# ---- GPU -----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pb():
    pbm.set_sync_errors(True)
    yield pbm
    pbm.set_step_logging(False)
    pbm.engine.FORCE_ENGINE = None


def _logs(pb, many, n):
    return [pb.last_step_log(i) for i in range(n)] if many else [pb.last_step_log()]


def _run(pb, net, y0, t, target, engine, many, logging=True, rtol=1e-5, atol=1e-7, **kw):
    """Forward + backward on the GPU with the keyword arguments of odeint_adjoint(_many).  Returns y, adj_y0, the six
    .grad, forward and backward step logs (None when not logged) and the n_rhs of the last forward and backward solve."""
    saved = pb.engine.FORCE_ENGINE
    pb.engine.FORCE_ENGINE = engine
    pb.set_step_logging(logging)
    plist = list(net.parameters())
    try:
        net.zero_grad(set_to_none=True)
        y0g = y0.cuda().requires_grad_(True)
        solve = pb.odeint_adjoint_many if many else pb.odeint_adjoint
        y = solve(net, y0g, t, rtol=rtol, atol=atol, method="dopri5", **kw)
        flog = _logs(pb, many, y0.shape[0]) if logging else None
        fn = pb.engine.last_status()["n_rhs"]
        ys = y[:, 1:] if many else y[1:]
        ((ys - target.cuda()) ** 2).sum().backward()
        blog = _logs(pb, many, y0.shape[0]) if logging else None
        bn = pb.engine.last_status()["n_rhs"]
        return (y.detach().cpu(), y0g.grad.cpu(), [p.grad.detach().cpu().clone() for p in plist], flog, blog, fn, bn)
    finally:
        pb.set_step_logging(False)
        pb.engine.FORCE_ENGINE = saved


def _same(a, b, what):
    assert torch.equal(a[0], b[0]), (what, "y")
    assert torch.equal(a[1], b[1]), (what, "adj_y0")
    for i in range(6):
        assert torch.equal(a[2][i], b[2][i]), (what, NAMES[i])


def _copies(y0, t, target, many):
    """N copies of problem 0, so that every row / problem has the same Hairer estimate."""
    if not many:
        return y0, t, target
    n = y0.shape[0]
    return (y0[:1].expand_as(y0).contiguous(), t[:1].expand_as(t).contiguous(), target[:1].expand_as(target).contiguous())


@pytest.mark.gpu
@pytest.mark.parametrize("e", ENGINES, ids=[_eid(e) for e in ENGINES])
def test_explicit_defaults_change_nothing(pb, e):
    engine, G, H, shape, many, times = e
    w, y0, t, target = _problem(G, H, shape, many, times, 41)
    net = make_net(pb, w)
    logging = not (engine == "resident" and many)
    ref = _run(pb, net, y0, t, target, engine, many, logging)
    got = _run(pb, net, y0, t, target, engine, many, logging, options=dict(DEFAULTS))
    _same(got, ref, _eid(e))
    assert got[3:] == ref[3:]


@pytest.mark.gpu
@pytest.mark.parametrize("e", ENGINES, ids=[_eid(e) for e in ENGINES])
def test_first_step_equal_to_hairer_changes_only_the_count(pb, e):
    """Forward over T = 3, backward over one interval (later intervals have estimates of their own): the first dt of a
    run without options passed back as first_step gives the same bits, one RHS evaluation fewer per solve."""
    engine, G, H, shape, many, _ = e
    for times, side in (((0.0, 0.1, 0.2), "forward"), ((0.0, 0.1), "backward")):
        w, y0, t, target = _problem(G, H, shape, many, times, 43)
        y0, t, target = _copies(y0, t, target, many)
        net = make_net(pb, w)
        probe = _run(pb, net, y0[:1] if engine == "resident" and many else y0,
                     t[:1] if engine == "resident" and many else t,
                     target[:1] if engine == "resident" and many else target, engine, many)
        h = (probe[3] if side == "forward" else probe[4])[0][0][1]
        logging = not (engine == "resident" and many)
        ref = _run(pb, net, y0, t, target, engine, many, logging)
        kw = dict(options=dict(first_step=h), adjoint_options={}) if side == "forward" else \
            dict(adjoint_options=dict(first_step=h))
        got = _run(pb, net, y0, t, target, engine, many, logging, **kw)
        _same(got, ref, (_eid(e), side))
        if logging:
            assert got[3] == ref[3] and got[4] == ref[4], (_eid(e), side)
        if side == "forward":
            assert (got[5], got[6]) == (ref[5] - 1, ref[6]), (_eid(e), side)
        else:
            assert (got[5], got[6]) == (ref[5], ref[6] - 1), (_eid(e), side)


def _oracle(w, y0, t, target, many, rtol, atol, opts):
    probs = [(y0[i], t[i], target[i]) for i in range(y0.shape[0])] if many else [(y0, t, target)]
    ys, adys, gsum, flogs, blogs = [], [], None, [], []
    for y0i, ti, tgi in probs:
        yr, flog = odeint_x(w, y0i, ti, rtol=rtol, atol=atol, **opts)
        gy = torch.zeros_like(yr)
        gy[1:] = 2.0 * (yr[1:] - tgi)
        ar, gr, blog = adjoint_backward_x(w, ti, yr, gy, rtol=rtol, atol=atol, **opts)
        ys.append(yr)
        adys.append(ar)
        gsum = gr if gsum is None else [a + b for a, b in zip(gsum, gr)]
        flogs.append(flog.steps)
        blogs.append(blog.steps)
    return (torch.stack(ys) if many else ys[0]), (torch.stack(adys) if many else adys[0]), gsum, flogs, blogs


def _counts_close(mine, ref, what):
    """The attempt and acceptance counts of assert_logs_close at the noise floor: accepted within max(1, 15 %), attempts
    within max(3, 40 %)."""
    acc_m, acc_r = sum(1 for x in mine if x[2]), sum(1 for x in ref if x[2])
    assert abs(acc_m - acc_r) <= max(1, int(0.15 * acc_r)), (what, "accepted", mine, ref)
    assert abs(len(mine) - len(ref)) <= max(3, int(0.4 * len(ref))), (what, "attempts", mine, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("e", ENGINES, ids=[_eid(e) for e in ENGINES])
def test_options_against_oracle(pb, e):
    """first_step at 1/4 and 20x of Hairer's estimate of the forward, and safety 0.8, ifactor 5, dfactor 0.5, passed in
    `options` and so inherited by the backward.  Resident and streaming run T = 3, rows T = 2.  The first attempt of
    every solve and backward interval has dt == first_step exactly, and at 20x the kernel rejects it where the oracle
    does.

    At 1/4 of Hairer's estimate the first attempts' error ratio is about 1e-4 (Hairer's step aims at 1e-2 of the
    tolerance, and the error scales with dt^5): fp32 rounding noise at rtol 1e-5.  The controller's next dt, a fifth root
    of that ratio, then differs from the oracle's by up to 30 % (observed on the 690-gene rows case), and the solutions
    follow different step sequences.  So for that case the logs are held to the noise-floor counts of
    assert_logs_close beyond the first attempt, and y, adj_y0 and the gradients to the rule of
    test_dopri5_seminorm_with_rejected_steps: no further from a float64 solve at rtol 1e-8 than 3x the fp32 oracle's own
    distance."""
    engine, G, H, shape, many, times = e
    rtol, atol = 1e-5, 1e-7
    w, y0, t, target = _problem(G, H, shape, many, times, 11)
    net = make_net(pb, w)
    logging = not (engine == "resident" and many)
    t0 = t[0] if many else t
    h = O.odeint(w, y0[0] if many else y0, t0, method="dopri5", rtol=rtol, atol=atol)[1].steps[0][1]
    rejected = False
    for opts in (dict(first_step=h / 4), dict(first_step=20 * h), dict(safety=0.8, ifactor=5.0, dfactor=0.5)):
        what = (_eid(e), opts)
        noise = opts.get("first_step") == h / 4
        got = _run(pb, net, y0, t, target, engine, many, logging, rtol=rtol, atol=atol, options=dict(opts))
        y_r, a_r, g_r, fl_r, bl_r = _oracle(w, y0, t, target, many, rtol, atol, opts)
        if noise:
            wd = O.Weights(*[p.double() for p in w.as_list()])
            y64, a64, g64, _, _ = _oracle(wd, y0.double(), t, target.double(), many, 1e-8, 1e-10, {})
            assert rel_l2(got[0], y64) <= 3 * rel_l2(y_r, y64) + 2e-7, (what, rel_l2(got[0], y64), rel_l2(y_r, y64))
            assert rel_l2(got[1], a64) <= 3 * rel_l2(a_r, a64) + 5e-6, (what, rel_l2(got[1], a64), rel_l2(a_r, a64))
            for i in range(6):
                assert rel_l2(got[2][i], g64[i]) <= 3 * rel_l2(g_r[i], g64[i]) + 5e-6, \
                    (what, NAMES[i], rel_l2(got[2][i], g64[i]), rel_l2(g_r[i], g64[i]))
        else:
            assert rel_l2(got[0], y_r) < 1e-5, what
            assert rel_l2(got[1], a_r) < 1e-5, (what, rel_l2(got[1], a_r))
            for i in range(6):
                assert rel_l2(got[2][i], g_r[i]) < 5e-5, (what, NAMES[i], rel_l2(got[2][i], g_r[i]))
        if not logging:
            continue
        fs = opts.get("first_step")
        for i, (fm, fr, bm, br) in enumerate(zip(got[3], fl_r, got[4], bl_r)):
            ti = t[i] if many else t
            if fs is not None:
                assert fm[0][1] == fs and fr[0][1] == fs, what
                starts_m, starts_r = interval_starts(bm, ti), interval_starts(br, ti)
                assert all(s[1] == fs for s in starts_m + starts_r), what
                assert [s[2] for s in starts_m] == [s[2] for s in starts_r], what
                assert fm[0][2] == fr[0][2], what
                rejected = rejected or not fr[0][2]
            if noise:
                _counts_close(fm, fr, "%s fwd %d" % (what, i))
                _counts_close(bm, br, "%s bwd %d" % (what, i))
            else:
                assert_logs_close(fm, fr, 0.25, "%s fwd %d" % (what, i), first_rtol=0.0 if fs else 1e-4)
                assert_logs_close(bm, br, 0.25, "%s bwd %d" % (what, i), first_rtol=0.0 if fs else 1e-4)
    if logging:
        assert rejected, "20x Hairer's estimate is accepted by the oracle: the case does not exercise dfactor"


@pytest.mark.gpu
def test_per_sample_loop_with_options_matches_many(pb):
    """The literal loop of training_step with the options: the deferred backward gives bit for bit what
    odeint_adjoint_many gives."""
    G, H, N = 690, 40, 6
    w = O.make_weights(G, H, 21, dense=True, neg_mult_frac=0.2)
    gen = torch.Generator().manual_seed(22)
    y0 = torch.rand(N, 1, G, generator=gen)
    t = torch.rand(N, 1, generator=gen, dtype=torch.float64) + torch.tensor([0.0, 0.1], dtype=torch.float64)
    target = torch.rand(N, 1, G, generator=gen)
    net = make_net(pb, w)
    params = list(net.parameters())
    for opts in (dict(first_step=0.01), dict(first_step=0.02, safety=0.8, ifactor=5.0, dfactor=0.5)):
        net.zero_grad(set_to_none=True)
        preds = [pb.odeint_adjoint(net, y0[i].cuda(), t[i], method="dopri5", options=opts)[1] for i in range(N)]
        torch.mean((torch.stack(preds) - target.cuda()) ** 2).backward()
        loop = [p.grad.clone() for p in params]
        net.zero_grad(set_to_none=True)
        y = pb.odeint_adjoint_many(net, y0.cuda(), t, method="dopri5", options=opts)
        torch.mean((y[:, 1] - target.cuda()) ** 2).backward()
        for i in range(6):
            assert torch.equal(loop[i], params[i].grad), (opts, NAMES[i])


@pytest.mark.gpu
def test_phx_solve_refuses_invalid_step_control(pb):
    """phx_solve refuses a negative, NaN or infinite value in any of the four fields, and a nonzero one with a method
    other than dopri5, on every engine and direction; the valid requests next to them run."""
    from phoenix_b200 import _lib
    rq = _Requests(pb)
    for engine in ("resident", "rows", "stream"):
        for adjoint in (0, 1):
            for key in ("first_step", "safety", "ifactor", "dfactor"):
                for bad in (-0.1, float("nan"), float("inf"), -float("inf")):
                    assert rq.solve(engine, adjoint, method=3, **{key: bad}) == -1, (engine, adjoint, key, bad)
                    assert key in _lib.last_error(), (engine, adjoint, key)
                for method in (0, 1, 2):
                    assert rq.solve(engine, adjoint, method=method, **{key: 0.5}) == -1, (engine, adjoint, key, method)
                    assert key in _lib.last_error(), (engine, adjoint, key)
            assert rq.solve(engine, adjoint, method=3, first_step=0.01, safety=0.8, ifactor=5.0, dfactor=0.5) == 0, \
                (engine, adjoint, _lib.last_error())
            torch.cuda.synchronize()
