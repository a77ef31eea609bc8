"""Frozen parameters and explicit ``adjoint_params`` in ``odeint_adjoint`` (adjoint.py:185-193).

The adjoint set S is the members of ``adjoint_params`` (default: the six ODENet parameters) that require grad.  The
backward integrates, puts in the error norm and returns only the cotangents of S; the forward solve and adj_y0's
dependence on the state do not change.  CPU tests pin the oracle and the host logic; GPU tests hold every adjoint
engine (resident, resident many, rows at 4 / 2 / 1 rows per pass, streaming) to the oracle run with the same S."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import phoenix_b200 as pbm
from phoenix_b200 import parallel
from phoenix_b200.torchdiffeq import _api
from oracle import phoenix_oracle as O
from golden_util import assert_logs_close, rel_l2
from test_gpu_placements import CASES, _case_id, _check_tier, _inputs, make_net

NAMES = O.PARAM_ORDER
# S = {m}, all but Wa, {Wa, m}, {bs}; the fourth is given in reverse reference order
SUBSETS = [(0,), (0, 1, 2, 3, 4), (5, 0), (4,)]


# ---- oracle (CPU) ----------------------------------------------------------------------------------------------------------
def adjoint_backward_s(w, t, y, grad_y, method=None, rtol=1e-7, atol=1e-9, params=None):
    """``oracle.phoenix_oracle.adjoint_backward`` restricted to the adjoint set S (``params``: indices in reference order,
    None = all six): the augmented state is ``[vjp_t, y, adj_y, *S]`` (adjoint.py:86-151) and its norm
    ``max(RMS(vjp_t), RMS(y), RMS(adj_y), RMS(concatenation of S))`` (adjoint.py:72-78).  With S empty the parameter
    block is absent: the reference's ``_rms_norm`` of an empty tensor is NaN, and the Python ``max`` of adjoint.py:78
    keeps its current value when a later argument is NaN.  Returns (adj_y0, [6 grads, None outside S], StepLog)."""
    log = O.StepLog([])
    shape = y.shape[1:]
    N = y[0].numel()
    sel = list(range(6)) if params is None else sorted(set(int(i) for i in params))
    allp = w.as_list()
    psz = [allp[i].numel() for i in sel]
    P = sum(psz)
    norm = O.block_max_rms([1, N, N, P] if P else [1, N, N])

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


def _oracle_problem(G=64, H=8, method="dopri5"):
    w = O.make_weights(G, H, 3, dense=True, neg_mult_frac=0.2)
    gen = torch.Generator().manual_seed(4)
    y0 = torch.rand(1, G, generator=gen)
    t = torch.tensor([0.0, 0.3, 0.6], dtype=torch.float64)
    target = torch.rand(2, 1, G, generator=gen)
    y, _ = O.odeint(w, y0, t, method=method)
    gy = torch.zeros_like(y)
    gy[1:] = 2.0 * (y[1:] - target)   # loss = sum of squares: the cotangents are large enough for the theta block to matter
    return w, t, y, gy


@pytest.mark.parametrize("method", ["euler", "midpoint", "rk4"])
def test_oracle_fixed_grid_subset_is_exact(method):
    """The norm is never used on a fixed grid: adj_y0 and the S-cotangents equal the all-six backward bit for bit."""
    w, t, y, gy = _oracle_problem(method=method)
    a0, g0, _ = adjoint_backward_s(w, t, y, gy, method=method)
    for S in SUBSETS + [()]:
        a, g, _ = adjoint_backward_s(w, t, y, gy, method=method, params=S)
        assert torch.equal(a, a0), S
        for i in range(6):
            if i in S:
                assert torch.equal(g[i], g0[i]), (S, NAMES[i])
            else:
                assert g[i] is None, (S, NAMES[i])


@pytest.mark.parametrize("S", [(0,), ()])
def test_oracle_dopri5_first_step_sees_the_mask(S):
    """While theta is zero its block is scaled by atol and dominates d1 of Hairer's initial step: the first backward dt
    with S = {m} or S = {} differs from the all-six one by far more than the 1e-4 first-step tolerance."""
    w, t, y, gy = _oracle_problem()
    _, _, log_all = adjoint_backward_s(w, t, y, gy, method="dopri5")
    _, g, log = adjoint_backward_s(w, t, y, gy, method="dopri5", params=S)
    dt_all, dt = log_all.steps[0][1], log.steps[0][1]
    assert abs(dt - dt_all) > 1e-2 * abs(dt_all), (dt, dt_all)
    assert all((g[i] is None) == (i not in S) for i in range(6))


def test_oracle_all_six_is_the_oracle():
    """With S = all six the restriction is the oracle's own backward, bit for bit (steps included)."""
    w, t, y, gy = _oracle_problem()
    a0, g0, l0 = O.adjoint_backward(w, t, y, gy, method="dopri5")
    a1, g1, l1 = adjoint_backward_s(w, t, y, gy, method="dopri5", params=range(6))
    assert torch.equal(a0, a1) and all(torch.equal(x, z) for x, z in zip(g0, g1)) and l0.steps == l1.steps


# ---- host logic (CPU) ------------------------------------------------------------------------------------------------------
def _cpu_net():
    torch.manual_seed(0)
    return pbm.ODENet("cpu", 12, neurons=4)


def test_mask_from_requires_grad_and_adjoint_params():
    net = _cpu_net()
    params = list(net.parameters())
    assert _api._adjoint_mask(net, None)[1] == 0x3F
    params[3].requires_grad_(False)                      # Ws frozen
    assert _api._adjoint_mask(net, None)[1] == 0x3F & ~(1 << 3)
    # explicit subsets: matched by identity, any order; a frozen member is still left out
    assert _api._adjoint_mask(net, [params[5], params[0]])[1] == (1 << 5) | 1
    assert _api._adjoint_mask(net, (params[3], params[4]))[1] == 1 << 4
    assert _api._adjoint_mask(net, ())[1] == 0
    assert _api._adjoint_mask(net, iter(params[::-1]))[1] == 0x3F & ~(1 << 3)


def test_adjoint_params_rejects_foreign_and_duplicate_tensors():
    net = _cpu_net()
    params = list(net.parameters())
    y0 = torch.rand(1, 12)
    t = torch.tensor([0.0, 1.0])
    for bad in ([params[0], params[0]], [torch.zeros(1, 12, requires_grad=True)], [params[1].detach()], [params[2], 3]):
        with pytest.raises(NotImplementedError):
            pbm.odeint_adjoint(net, y0, t, adjoint_params=bad)
        with pytest.raises(NotImplementedError):
            pbm.odeint_adjoint_many(net, y0.unsqueeze(0), t.unsqueeze(0), adjoint_params=bad)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    net = pbm.ODENet("cpu", 12, neurons=4)
    params = list(net.parameters())
    params[3].requires_grad_(False)                      # Ws frozen: its .grad stays None through the collective
    for i, p in enumerate(params):
        p.grad = None if i == 3 else torch.full_like(p, float((i + 1) * (rank + 1)))
    parallel.allreduce_grads(net, average=False)
    ok = params[3].grad is None
    ok = ok and all(torch.equal(p.grad, torch.full_like(p, float((i + 1) * 3))) for i, p in enumerate(params) if i != 3)
    if rank == 0:
        with open(out, "w") as fh:
            fh.write("%d" % int(ok))
    dist.destroy_process_group()


def test_allreduce_keeps_frozen_grad_none_world2(tmp_path):
    out = os.path.join(str(tmp_path), "res.txt")
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    assert open(out).read() == "1"


# ---- GPU -----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pb():
    pbm.set_sync_errors(True)
    yield pbm
    pbm.set_step_logging(False)
    pbm.engine.FORCE_ENGINE = None


def _backward(pb, net, y0, t, target, method, S, engine, many, explicit, rtol=1e-7, atol=1e-9):
    """One forward + backward on the GPU with adjoint set S (None: all six) given through requires_grad or, with
    `explicit`, through adjoint_params (in the order S lists them).  Returns y, adj_y0, the six .grad (None allowed)."""
    params = list(net.parameters())
    saved = pb.engine.FORCE_ENGINE
    pb.engine.FORCE_ENGINE = engine
    try:
        net.zero_grad(set_to_none=True)
        for i, p in enumerate(params):
            p.requires_grad_(S is None or explicit or i in S)
        kw = {}
        if explicit and S is not None:
            kw["adjoint_params"] = [params[i] for i in S]
        y0g = y0.cuda().requires_grad_(True)
        solve = pb.odeint_adjoint_many if many else pb.odeint_adjoint
        y = solve(net, y0g, t, rtol=rtol, atol=atol, method=method, **kw)
        ys = y[:, 1:] if many else y[1:]
        loss = ((ys - target.cuda()) ** 2).sum()
        loss.backward()
        return (y.detach().cpu(), y0g.grad.cpu(),
                [None if p.grad is None else p.grad.detach().cpu().clone() for p in params])
    finally:
        pb.engine.FORCE_ENGINE = saved
        for p in params:
            p.requires_grad_(True)


def _assert_subset_bits(full, sub, S, what):
    y0, a0, g0 = full
    y1, a1, g1 = sub
    assert torch.equal(y1, y0), (what, "y")
    assert torch.equal(a1, a0), (what, "adj_y0")
    for i in range(6):
        if i in S:
            assert g1[i] is not None and torch.equal(g1[i], g0[i]), (what, NAMES[i])
        else:
            assert g1[i] is None, (what, NAMES[i], "outside S")


ADJ_CASES = [c for c in CASES if c.adjoint]


@pytest.mark.gpu
@pytest.mark.parametrize("c", ADJ_CASES, ids=[_case_id(c) for c in ADJ_CASES])
def test_fixed_grid_subsets_bit_identical(pb, c):
    """Every adjoint placement class: adj_y0 and the S-cotangents equal the all-six call bit for bit, None outside S."""
    _check_tier(c)
    w, y0, t, target = _inputs(c, 31)
    net = make_net(pb, w)
    engine = "resident" if c.kernel == "resident" else "rows"
    many = c.kernel == "rows"
    full = _backward(pb, net, y0, t, target, c.method, None, engine, many, False)
    for k, S in enumerate(SUBSETS):
        sub = _backward(pb, net, y0, t, target, c.method, S, engine, many, explicit=k % 2 == 1)
        _assert_subset_bits(full, sub, S, (_case_id(c), S))


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["euler", "rk4"])
def test_fixed_grid_subsets_bit_identical_stream(pb, method):
    """The streaming engine on a 60-row batch (its contractions on the tensor cores)."""
    G, H, B = 1001, 100, 60
    w = O.make_weights(G, H, 7, dense=True, neg_mult_frac=0.2)
    gen = torch.Generator().manual_seed(8)
    y0 = torch.rand(B, G, generator=gen)
    t = torch.tensor([0.0, 0.05, 0.1])
    target = torch.rand(2, B, G, generator=gen)
    net = make_net(pb, w)
    full = _backward(pb, net, y0, t, target, method, None, "stream", False, False)
    for k, S in enumerate(SUBSETS + [()]):
        sub = _backward(pb, net, y0, t, target, method, S, "stream", False, explicit=k % 2 == 1)
        _assert_subset_bits(full, sub, S, ("stream", method, S))


# dopri5 against the fp32 oracle with the same S: (engine, G, H, y0 shape, many)
DOPRI = [
    ("resident", 350, 40, (1, 350), False),
    ("resident", 350, 40, (3, 1, 350), False),
    ("resident", 350, 40, (3, 2, 350), True),      # phx_solve_adjoint_many: several problems per launch
    ("rows", 690, 200, (5, 1, 690), True),         # 4 rows per pass
    ("rows", 13000, 129, (3, 1, 13000), True),     # 2 rows per pass
    ("rows", 16000, 100, (3, 1, 16000), True),     # 1 row per pass
    ("stream", 350, 40, (6, 350), False),
]
DOPRI_S = [(0,), (), (5, 0), (0, 1, 2, 3, 4)]
# Above the fp32 noise floor of the error estimate: at the default rtol 1e-7 the step sequence after the first step is
# set by rounding noise (the fp32 oracle and the fp64 one already differ by 26 % in the second dt with S = all but Wa)
RTOL, ATOL = 1e-5, 1e-7


def _dopri_id(d):
    return "%s-%dx%d-%s%s" % (d[0], d[1], d[2], "x".join(map(str, d[3])), "-many" if d[4] else "")


@pytest.mark.gpu
@pytest.mark.parametrize("d", DOPRI, ids=[_dopri_id(d) for d in DOPRI])
def test_dopri5_subsets_against_oracle(pb, d):
    engine, G, H, shape, many = d
    w = O.make_weights(G, H, 11, dense=True, neg_mult_frac=0.2)
    if G > 1000:
        w.Wp.mul_((1000.0 / G) ** 0.5)
        w.Ws.mul_((1000.0 / G) ** 0.5)
    gen = torch.Generator().manual_seed(12)
    y0 = torch.rand(*shape, generator=gen)
    # one output interval per problem, as in a training step (one time step per sample)
    times = torch.tensor([0.0, 0.1], dtype=torch.float64)
    if many:
        t = torch.rand(shape[0], 1, generator=gen, dtype=torch.float64) + times
        target = torch.rand(shape[0], 1, *shape[1:], generator=gen)
        probs = [(y0[i], t[i], target[i]) for i in range(shape[0])]
    else:
        t = times
        target = torch.rand(1, *shape, generator=gen)
        probs = [(y0, t, target)]
    net = make_net(pb, w)
    # the many-problems-per-launch path only runs without step logging
    logging = not (engine == "resident" and many)
    for k, S in enumerate(DOPRI_S):
        pb.set_step_logging(logging)
        try:
            y, ady, grads = _backward(pb, net, y0, t, target, "dopri5", S, engine, many, explicit=k % 2 == 1,
                                      rtol=RTOL, atol=ATOL)
            blogs = [pb.last_step_log(i) for i in range(len(probs))] if (logging and many) else \
                [pb.last_step_log()] if logging else None
        finally:
            pb.set_step_logging(False)
        ys, adys, gsum, refl = [], [], None, []
        for y0i, ti, tgi in probs:
            yr, _ = O.odeint(w, y0i, ti, method="dopri5", rtol=RTOL, atol=ATOL)
            gy = torch.zeros_like(yr)
            gy[1:] = 2.0 * (yr[1:] - tgi)
            ar, gr, blog = adjoint_backward_s(w, ti, yr, gy, method="dopri5", params=S, rtol=RTOL, atol=ATOL)
            ys.append(yr)
            adys.append(ar)
            gsum = gr if gsum is None else [a if a is None else a + b for a, b in zip(gsum, gr)]
            refl.append(blog.steps)
        y_ref = torch.stack(ys) if many else ys[0]
        ady_ref = torch.stack(adys) if many else adys[0]
        what = (_dopri_id(d), S)
        assert rel_l2(y, y_ref) < 1e-5, what
        assert rel_l2(ady, ady_ref) < 1e-5, (what, rel_l2(ady, ady_ref))
        for i in range(6):
            if i in S:
                assert rel_l2(grads[i], gsum[i]) < 5e-5, (what, NAMES[i], rel_l2(grads[i], gsum[i]))
            else:
                assert grads[i] is None, (what, NAMES[i])
        if blogs is not None:
            for i, (mine, ref) in enumerate(zip(blogs, refl)):
                assert_logs_close(mine, ref, 0.25, "%s bwd %d" % (what, i))


@pytest.mark.gpu
def test_per_sample_loop_with_frozen_parameter_matches_many(pb):
    """The literal loop of training_step with Ws frozen: the deferred backward still solves all sweeps in one rows call
    and gives bit for bit what odeint_adjoint_many gives with the same S."""
    G, H, N = 690, 40, 6
    w = O.make_weights(G, H, 21, dense=True, neg_mult_frac=0.2)
    gen = torch.Generator().manual_seed(22)
    y0 = torch.rand(N, 1, G, generator=gen)
    t = torch.rand(N, 1, generator=gen, dtype=torch.float64) + torch.tensor([0.0, 0.1], dtype=torch.float64)
    target = torch.rand(N, 1, G, generator=gen)
    net = make_net(pb, w)
    params = list(net.parameters())
    params[3].requires_grad_(False)
    try:
        for method in ("rk4", "dopri5"):
            net.zero_grad(set_to_none=True)
            preds = [pb.odeint_adjoint(net, y0[i].cuda(), t[i], method=method)[1] for i in range(N)]
            torch.mean((torch.stack(preds) - target.cuda()) ** 2).backward()
            loop = [None if p.grad is None else p.grad.clone() for p in params]
            net.zero_grad(set_to_none=True)
            y = pb.odeint_adjoint_many(net, y0.cuda(), t, method=method)
            torch.mean((y[:, 1] - target.cuda()) ** 2).backward()
            assert loop[3] is None and params[3].grad is None
            for i in (0, 1, 2, 4, 5):
                assert torch.equal(loop[i], params[i].grad), (method, NAMES[i])
    finally:
        params[3].requires_grad_(True)
