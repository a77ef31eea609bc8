"""Seminorm error control in the adjoint backward: ``adjoint_options=dict(norm="seminorm")``.

The seminorm (Kidger, Chen & Lyons, "Hey, that's not an ODE", 2021) is the backward's mixed error norm without the
parameter-cotangent block: ``max(RMS(vjp_t), RMS(y), RMS(adj_y))``, in Hairer's initial step and in every error ratio.
The cotangents of the adjoint set S are still integrated.  CPU tests pin the oracle and the host logic.  GPU tests check
on every adjoint engine (resident, resident many, rows at 4 / 2 / 1 rows per pass, streaming) that the seminorm with S =
all six steps exactly like the default norm with S empty, that fixed grids do not notice the option, and that dopri5
follows the oracle under the seminorm."""
import pytest
import torch

import phoenix_b200 as pbm
from phoenix_b200.torchdiffeq import _api
from oracle import phoenix_oracle as O
from golden_util import assert_logs_close, rel_l2
from test_gpu_adjoint_params import _oracle_problem, adjoint_backward_s
from test_gpu_placements import A, CASES, R, W, _case_id, _check_tier, _inputs, _set_knobs, make_net

NAMES = O.PARAM_ORDER
SEMI = {"norm": "seminorm"}


# ---- oracle (CPU) ----------------------------------------------------------------------------------------------------------
def adjoint_backward_semi(w, t, y, grad_y, method=None, rtol=1e-7, atol=1e-9, params=None):
    """``adjoint_backward_s`` under the seminorm: the augmented state is still ``[vjp_t, y, adj_y, *S]``, but its norm
    is ``block_max_rms([1, N, N])`` of the first 1 + 2N entries, for the initial step and the error ratio alike.
    Returns (adj_y0, [6 grads, None outside S], StepLog)."""
    log = O.StepLog([])
    shape = y.shape[1:]
    N = y[0].numel()
    sel = list(range(6)) if params is None else sorted(set(int(i) for i in params))
    allp = w.as_list()
    psz = [allp[i].numel() for i in sel]
    P = sum(psz)
    head = O.block_max_rms([1, N, N])

    def norm(x):
        return head(x[:1 + 2 * N])

    def aug_reversed(tt, z):
        f, ybar, pbar = O.rhs_vjp(w, z[1:1 + N].reshape(shape), -z[1 + N:1 + 2 * N].reshape(shape))
        return -torch.cat([torch.zeros(1, dtype=z.dtype), f.reshape(-1), ybar.reshape(-1)]
                          + [pbar[i].reshape(-1) for i in sel])

    with torch.no_grad():
        adj_y = grad_y[-1].clone()
        adj_p = torch.zeros(P, dtype=y.dtype)
        cur_y = y[-1]
        for i in range(len(t) - 1, 0, -1):
            z0 = torch.cat([torch.zeros(1, dtype=y.dtype), cur_y.reshape(-1), adj_y.reshape(-1), adj_p])
            z = O._solve(aug_reversed, z0, -t[i - 1:i + 1].flip(0), method, rtol, atol, norm, log)[1]
            adj_p = z[1 + 2 * N:]
            cur_y = y[i - 1]
            adj_y = z[1 + N:1 + 2 * N].reshape(shape) + grad_y[i - 1]
        grads, lo = [None] * 6, 0
        for i, n in zip(sel, psz):
            grads[i] = adj_p[lo:lo + n].reshape(allp[i].shape)
            lo += n
    return adj_y, grads, log


@pytest.mark.parametrize("method", ["euler", "midpoint", "rk4"])
def test_oracle_fixed_grid_ignores_the_seminorm(method):
    w, t, y, gy = _oracle_problem(method=method)
    a0, g0, _ = adjoint_backward_s(w, t, y, gy, method=method)
    a1, g1, _ = adjoint_backward_semi(w, t, y, gy, method=method)
    assert torch.equal(a0, a1)
    assert all(torch.equal(x, z) for x, z in zip(g0, g1))


def test_oracle_seminorm_steps_like_the_empty_adjoint_set():
    """The seminorm with S = all six steps like the default norm with S empty: the y / adj_y algebra never reads theta.
    adj_y0 and the accept pattern agree bit for bit; a dt may differ in the last bits, because CPU BLAS rounds the fp32
    error combination differently for the longer augmented vector."""
    w, t, y, gy = _oracle_problem()
    a0, _, l0 = adjoint_backward_s(w, t, y, gy, method="dopri5", params=())
    a1, g1, l1 = adjoint_backward_semi(w, t, y, gy, method="dopri5")
    assert torch.equal(a0, a1)
    assert [s[2] for s in l0.steps] == [s[2] for s in l1.steps]
    for s0, s1 in zip(l0.steps, l1.steps):
        assert abs(s1[1] - s0[1]) <= 1e-6 * abs(s0[1]), (s0, s1)
    assert all(g is not None for g in g1)
    # ... and it is not the default norm with S = all six (whose theta block sets the first backward dt)
    _, _, lall = adjoint_backward_s(w, t, y, gy, method="dopri5")
    assert len(lall.steps) != len(l1.steps) or lall.steps[0][1] != l1.steps[0][1]


# ---- host logic (CPU) ------------------------------------------------------------------------------------------------------
def _cpu_net():
    torch.manual_seed(0)
    return pbm.ODENet("cpu", 12, neurons=4)


def _captured_adj(monkeypatch, many, **kw):
    """The ``adj`` tuple (method, rtol, atol, max_steps, mask) an entry point hands its autograd node."""
    got = {}

    def fake_apply(*args):
        got["adj"] = args[7]
        return None

    cls = _api.OdeintAdjointManyMethod if many else _api.OdeintAdjointMethod
    monkeypatch.setattr(cls, "apply", fake_apply)
    net = _cpu_net()
    y0 = torch.rand(1, 12)
    t = torch.tensor([0.0, 1.0])
    if many:
        pbm.odeint_adjoint_many(net, y0.unsqueeze(0), t.unsqueeze(0), method="dopri5", **kw)
    else:
        pbm.odeint_adjoint(net, y0, t, method="dopri5", **kw)
    return got["adj"]


@pytest.mark.parametrize("many", [False, True])
def test_seminorm_option_sets_the_norm_bit(monkeypatch, many):
    assert _captured_adj(monkeypatch, many)[4] == 0x3F
    assert _captured_adj(monkeypatch, many, adjoint_options=SEMI)[4] == 0x3F | 0x40
    assert _captured_adj(monkeypatch, many, adjoint_options=SEMI, adjoint_params=())[4] == 0x40
    # the other adjoint options are still honoured next to it
    adj = _captured_adj(monkeypatch, many, adjoint_options=dict(norm="seminorm", max_num_steps=7))
    assert adj[3] == 7 and adj[4] == 0x7F


@pytest.mark.parametrize("many", [False, True])
def test_other_norms_are_refused(many):
    net = _cpu_net()
    y0 = torch.rand(1, 12)
    t = torch.tensor([0.0, 1.0])
    solve = (lambda **kw: pbm.odeint_adjoint_many(net, y0.unsqueeze(0), t.unsqueeze(0), **kw)) if many else \
        (lambda **kw: pbm.odeint_adjoint(net, y0, t, **kw))
    for bad in (lambda x: x.abs().max(), "rms", "max", None):
        with pytest.raises(NotImplementedError, match="seminorm"):
            solve(adjoint_options={"norm": bad})
    with pytest.raises(NotImplementedError):   # the forward solve takes no norm, as before
        solve(options={"norm": "seminorm"})


class _Ctx:
    """Stands in for an autograd context (the live-node registry keeps weak references to it)."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


def test_deferred_group_key_includes_the_norm(monkeypatch):
    monkeypatch.setattr(_api, "DEFER_ADJOINT", True)
    net = _cpu_net()
    y0 = torch.rand(1, 12)
    keys = []
    for mask in (0x3F, 0x7F, 0x40):
        ctx = _Ctx(needs_input_grad=(False,) * 9 + (True,) * 6)
        _api._register_node(ctx, net, y0, [0.0, 1.0], True, ("dopri5", 1e-7, 1e-9, 100, mask))
        keys.append(ctx.group)
    assert keys[0] is not None and keys[1] is not None and keys[0] != keys[1]
    assert keys[2] is None   # an empty adjoint set is no deferred node, whatever the norm


@pytest.mark.parametrize("many", [False, True])
def test_empty_set_with_seminorm_needs_no_backward(monkeypatch, many):
    def boom(*a, **k):
        raise AssertionError("the backward ran")

    monkeypatch.setattr(_api.engine, "solve_adjoint", boom)
    monkeypatch.setattr(_api.engine, "solve_adjoint_many", boom)
    ctx = _Ctx(saved_tensors=(torch.zeros(2, 1, 12),), adj=("dopri5", 1e-7, 1e-9, 100, 0x40),
                                needs_input_grad=(False,) * 15, group=None)
    cls = _api.OdeintAdjointManyMethod if many else _api.OdeintAdjointMethod
    assert cls.backward(ctx, torch.zeros(2, 1, 12)) == (None,) * 15


# ---- GPU -----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pb():
    pbm.set_sync_errors(True)
    yield pbm
    pbm.set_step_logging(False)
    pbm.engine.FORCE_ENGINE = None


def _backward(pb, net, y0, t, target, method, engine, many, semi, params=None, rtol=1e-5, atol=1e-7, logging=True):
    """One forward + backward on the GPU.  ``params``: adjoint_params as indices (None: all six); ``semi``: the seminorm.
    Returns y, adj_y0, the six .grad (None allowed) and the backward step logs (None when not logged)."""
    plist = list(net.parameters())
    saved = pb.engine.FORCE_ENGINE
    pb.engine.FORCE_ENGINE = engine
    pb.set_step_logging(logging)
    try:
        net.zero_grad(set_to_none=True)
        kw = {}
        if params is not None:
            kw["adjoint_params"] = [plist[i] for i in params]
        if semi:
            kw["adjoint_options"] = SEMI
        y0g = y0.cuda().requires_grad_(True)
        solve = pb.odeint_adjoint_many if many else pb.odeint_adjoint
        y = solve(net, y0g, t, rtol=rtol, atol=atol, method=method, **kw)
        ys = y[:, 1:] if many else y[1:]
        ((ys - target.cuda()) ** 2).sum().backward()
        logs = None
        if logging:
            logs = [pb.last_step_log(i) for i in range(y0.shape[0])] if many else [pb.last_step_log()]
        return (y.detach().cpu(), y0g.grad.cpu(),
                [None if p.grad is None else p.grad.detach().cpu().clone() for p in plist], logs)
    finally:
        pb.set_step_logging(False)
        pb.engine.FORCE_ENGINE = saved


def _problem(G, H, shape, many, times, seed):
    w = O.make_weights(G, H, seed, dense=True, neg_mult_frac=0.2)
    if G > 1000:
        w.Wp.mul_((1000.0 / G) ** 0.5)
        w.Ws.mul_((1000.0 / G) ** 0.5)
    gen = torch.Generator().manual_seed(seed + 1)
    y0 = torch.rand(*shape, generator=gen)
    times = torch.tensor(times, dtype=torch.float64)
    if many:
        t = torch.rand(shape[0], 1, generator=gen, dtype=torch.float64) + times
        target = torch.rand(shape[0], len(times) - 1, *shape[1:], generator=gen)
    else:
        t = times
        target = torch.rand(len(times) - 1, *shape, generator=gen)
    return w, y0, t, target


# (engine, G, H, y0 shape, many, output times).  The rows engine gets one output interval per problem (DESIGN 8).
ENGINES = [
    ("resident", 350, 40, (1, 350), False, (0.0, 0.1, 0.2)),
    ("resident", 350, 40, (3, 2, 350), True, (0.0, 0.1, 0.2)),    # phx_solve_adjoint_many
    ("rows", 690, 200, (5, 1, 690), True, (0.0, 0.1)),            # 4 rows per pass
    ("rows", 13000, 129, (3, 1, 13000), True, (0.0, 0.1)),        # 2 rows per pass
    ("rows", 16000, 100, (3, 1, 16000), True, (0.0, 0.1)),        # 1 row per pass
    ("stream", 350, 40, (6, 350), False, (0.0, 0.1, 0.2)),
]


def _eid(e):
    return "%s-%dx%d-%s%s" % (e[0], e[1], e[2], "x".join(map(str, e[3])), "-many" if e[4] else "")


@pytest.mark.gpu
@pytest.mark.parametrize("e", ENGINES, ids=[_eid(e) for e in ENGINES])
def test_seminorm_steps_like_the_empty_adjoint_set(pb, e):
    """No tolerance: the y / adj_y stage algebra never reads theta, and the kernels' reductions keep the theta sums in
    slots of their own, so the seminorm with S = all six gives the adj_y0 and the step log of the default norm with S
    empty bit for bit."""
    engine, G, H, shape, many, times = e
    w, y0, t, target = _problem(G, H, shape, many, times, 41)
    net = make_net(pb, w)
    logging = not (engine == "resident" and many)   # the many-problems-per-launch path logs no steps
    y0_, a0, g0, l0 = _backward(pb, net, y0, t, target, "dopri5", engine, many, False, params=(), logging=logging)
    y1, a1, g1, l1 = _backward(pb, net, y0, t, target, "dopri5", engine, many, True, logging=logging)
    assert torch.equal(y1, y0_)
    assert torch.equal(a1, a0)
    assert all(g is None for g in g0) and all(g is not None for g in g1)
    if logging:
        assert l1 == l0
        assert sum(len(x) for x in l1) > 0


ADJ_CASES = [c for c in CASES if c.adjoint]


@pytest.mark.gpu
@pytest.mark.parametrize("c", ADJ_CASES, ids=[_case_id(c) for c in ADJ_CASES])
def test_fixed_grid_ignores_the_seminorm(pb, c):
    """Every adjoint placement class: a fixed grid uses no norm, so every output equals the default call bit for bit."""
    _check_tier(c)
    w, y0, t, target = _inputs(c, 37)
    net = make_net(pb, w)
    engine = "resident" if c.kernel == "resident" else "rows"
    many = c.kernel == "rows"
    for params in (None, (5, 0)):
        y0_, a0, g0, _ = _backward(pb, net, y0, t, target, c.method, engine, many, False, params, logging=False)
        y1, a1, g1, _ = _backward(pb, net, y0, t, target, c.method, engine, many, True, params, logging=False)
        assert torch.equal(y1, y0_) and torch.equal(a1, a0), (_case_id(c), params)
        for i in range(6):
            assert (g0[i] is None and g1[i] is None) or torch.equal(g1[i], g0[i]), (_case_id(c), params, NAMES[i])


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["euler", "midpoint", "rk4"])
def test_fixed_grid_ignores_the_seminorm_stream(pb, method):
    w, y0, t, target = _problem(1001, 100, (60, 1001), False, (0.0, 0.05, 0.1), 8)
    net = make_net(pb, w)
    ref = _backward(pb, net, y0, t, target, method, "stream", False, False, logging=False)
    got = _backward(pb, net, y0, t, target, method, "stream", False, True, logging=False)
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    assert all(torch.equal(a, b) for a, b in zip(got[2], ref[2]))


def _oracle(w, y0, t, target, many, params, rtol, atol):
    """fp32 oracle under the seminorm: y, adj_y0, the S-gradients summed over the problems, backward step logs."""
    probs = [(y0[i], t[i], target[i]) for i in range(y0.shape[0])] if many else [(y0, t, target)]
    ys, adys, gsum, logs = [], [], None, []
    for y0i, ti, tgi in probs:
        yr, _ = O.odeint(w, y0i, ti, method="dopri5", rtol=rtol, atol=atol)
        gy = torch.zeros_like(yr)
        gy[1:] = 2.0 * (yr[1:] - tgi)
        ar, gr, blog = adjoint_backward_semi(w, ti, yr, gy, method="dopri5", params=params, rtol=rtol, atol=atol)
        ys.append(yr)
        adys.append(ar)
        gsum = gr if gsum is None else [a if a is None else a + b for a, b in zip(gsum, gr)]
        logs.append(blog.steps)
    return (torch.stack(ys) if many else ys[0]), (torch.stack(adys) if many else adys[0]), gsum, logs


def _check_against_oracle(got, ref, S, what):
    y, ady, grads, logs = got
    y_ref, ady_ref, g_ref, logs_ref = ref
    assert rel_l2(y, y_ref) < 1e-5, what
    assert rel_l2(ady, ady_ref) < 1e-5, (what, rel_l2(ady, ady_ref))
    for i in range(6):
        if i in S:
            assert rel_l2(grads[i], g_ref[i]) < 5e-5, (what, NAMES[i], rel_l2(grads[i], g_ref[i]))
        else:
            assert grads[i] is None, (what, NAMES[i])
    if logs is not None:
        for i, (mine, r) in enumerate(zip(logs, logs_ref)):
            assert_logs_close(mine, r, 0.25, "%s bwd %d" % (what, i))


@pytest.mark.gpu
@pytest.mark.parametrize("e", ENGINES, ids=[_eid(e) for e in ENGINES])
def test_dopri5_seminorm_against_oracle(pb, e):
    """Tolerances of test_dopri5_subsets_against_oracle, S = all six and S = {Wa, m}."""
    engine, G, H, shape, many, times = e
    rtol, atol = 1e-5, 1e-7
    w, y0, t, target = _problem(G, H, shape, many, times, 11)
    net = make_net(pb, w)
    logging = not (engine == "resident" and many)
    for S in ((0, 1, 2, 3, 4, 5), (5, 0)):
        got = _backward(pb, net, y0, t, target, "dopri5", engine, many, True, params=S, rtol=rtol, atol=atol,
                        logging=logging)
        _check_against_oracle(got, _oracle(w, y0, t, target, many, S, rtol, atol), S, (_eid(e), S))


# (case, PHX_MIN_GENES_PER_CTA, output times): the ring-tier inputs of test_gpu_placements, where the backward rejects
# attempts -- what the seminorm's theta pass, run after the accept decision, must get right.  One interval for rows.
REJECT = [
    (R(A, 1001, 129, 1, (4, 1, 0, 1), 1, method="dopri5"), "136", (0.0, 2.0, 5.0)),   # resident, WA ring
    (W(A, 1001, 100, 2, (4, 2, 1), method="dopri5"), "110", (0.0, 5.0)),               # rows, 1 row per pass
]


@pytest.mark.gpu
@pytest.mark.parametrize("c,gmin,times", REJECT, ids=["%s-gmin%s" % (_case_id(c), g) for c, g, _ in REJECT])
def test_dopri5_seminorm_with_rejected_steps(pb, monkeypatch, c, gmin, times):
    """Loose tolerances (rtol 1e-4, atol 1e-6), the rule of test_dopri5_ring_tiers: the kernel rejects backward attempts
    where the fp32 oracle does, its logs follow the oracle's to the noise-floor rule, and y, adj_y0 and the gradients are
    no further from a float64 solve at rtol 1e-8 (seminorm as well) than 3x the fp32 oracle's own distance."""
    _set_knobs(monkeypatch, pb, gmin)
    _check_tier(c)
    rtol, atol = 1e-4, 1e-6
    w, y0, t, target = _inputs(c, 5100 + c.H, times)
    net = make_net(pb, w)
    engine, many = ("resident", False) if c.kernel == "resident" else ("rows", True)
    S = (0, 1, 2, 3, 4, 5)
    y, ady, grads, logs = _backward(pb, net, y0, t, target, "dopri5", engine, many, True, rtol=rtol, atol=atol)
    y32, ady32, g32, logs32 = _oracle(w, y0, t, target, many, S, rtol, atol)
    wd = O.Weights(*[p.double() for p in w.as_list()])
    y64, ady64, g64, _ = _oracle(wd, y0.double(), t, target.double(), many, S, 1e-8, 1e-10)
    assert any(not s[2] for log in logs32 for s in log), "the oracle rejects no backward step"
    assert any(not s[2] for log in logs for s in log), "the oracle rejects a backward step, the kernel never does"
    # The first dt to 1e-3, not 1e-4: without the theta block (whose Gram norms are formed in double), d2 of Hairer's
    # initial step is the RMS of the difference of two fp32 RHS values h0 apart, and carries their rounding (1.5e-4
    # observed on the rows case).
    for i, (mine, ref) in enumerate(zip(logs, logs32)):
        assert_logs_close(mine, ref, 0.25, "%s bwd %d" % (_case_id(c), i), first_rtol=1e-3)
    assert rel_l2(y, y64) <= 3 * rel_l2(y32, y64) + 2e-7
    assert rel_l2(ady, ady64) <= 3 * rel_l2(ady32, ady64) + 5e-6, (rel_l2(ady, ady64), rel_l2(ady32, ady64))
    for i, (g, r32, r64) in enumerate(zip(grads, g32, g64)):
        assert rel_l2(g, r64) <= 3 * rel_l2(r32, r64) + 5e-6, (NAMES[i], rel_l2(g, r64), rel_l2(r32, r64))


@pytest.mark.gpu
def test_per_sample_loop_with_seminorm_matches_many(pb):
    """The literal loop of training_step under the seminorm: the deferred backward solves all sweeps in one rows call
    and gives bit for bit what odeint_adjoint_many gives with the seminorm."""
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
        preds = [pb.odeint_adjoint(net, y0[i].cuda(), t[i], method=method, adjoint_options=SEMI)[1] for i in range(N)]
        torch.mean((torch.stack(preds) - target.cuda()) ** 2).backward()
        loop = [p.grad.clone() for p in params]
        net.zero_grad(set_to_none=True)
        y = pb.odeint_adjoint_many(net, y0.cuda(), t, method=method, adjoint_options=SEMI)
        torch.mean((y[:, 1] - target.cuda()) ** 2).backward()
        for i in range(6):
            assert torch.equal(loop[i], params[i].grad), (method, NAMES[i])


@pytest.mark.gpu
def test_seminorm_gradient_accuracy(pb):
    """G = 350, H = 40 at the default tolerances (rtol 1e-7, atol 1e-9): the seminorm's gradients against a float64
    oracle solve at rtol 1e-10, next to the default norm's error on the same problem.  The seminorm takes fewer backward
    steps, so its error may be larger; it stays within 3x the default norm's error + 1e-6 (relative L2).  Observed on a
    B200 (1000 W): backward attempts 45 (default) and 47 (seminorm); relative L2 against float64 at most 3.06e-6
    (default, adj_y0) and 3.10e-6 (seminorm, adj_y0), the largest ratio seminorm / default 1.33 (bs)."""
    w, y0, t, target = _problem(350, 40, (1, 350), False, (0.0, 0.5, 1.0), 61)
    net = make_net(pb, w)
    default = _backward(pb, net, y0, t, target, "dopri5", "resident", False, False, rtol=1e-7, atol=1e-9)
    semi = _backward(pb, net, y0, t, target, "dopri5", "resident", False, True, rtol=1e-7, atol=1e-9)
    wd = O.Weights(*[p.double() for p in w.as_list()])
    y64, _ = O.odeint(wd, y0.double(), t, method="dopri5", rtol=1e-10, atol=1e-12)
    gy = torch.zeros_like(y64)
    gy[1:] = 2.0 * (y64[1:] - target.double())
    a64, g64, _ = O.adjoint_backward(wd, t, y64, gy, method="dopri5", rtol=1e-10, atol=1e-12)
    print("backward attempts: default %d, seminorm %d" % (len(default[3][0]), len(semi[3][0])))
    e_def = [rel_l2(a, r) for a, r in zip([default[1]] + default[2], [a64] + list(g64))]
    e_semi = [rel_l2(a, r) for a, r in zip([semi[1]] + semi[2], [a64] + list(g64))]
    for name, ed, es in zip(["adj_y0"] + list(NAMES), e_def, e_semi):
        print("%-16s default %.2e  seminorm %.2e" % (name, ed, es))
        assert es <= 3 * ed + 1e-6, (name, es, ed)
