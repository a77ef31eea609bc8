"""dopri5 on every engine against a float64 replay of the kernel's own step sequence.

At rtol 1e-7 the dopri5 error estimate is fp32 rounding noise, so the step sequence a solve takes depends on summation
order (DESIGN.md section 5): a kernel and an oracle that each choose their own steps can only be compared loosely.  Here
the oracle takes the steps the kernel logged (``O.Replay``: each attempt's dt and accept decision, forward and backward)
in float64.  What is left between the two is the kernel's fp32 rounding -- and its bugs -- so y, adj_y0, t.grad and the
gradients of the adjoint set S are held to the fp32 bar of ``test_gpu_placements`` at any rtol: relative L2 <= 1e-5 and
every element within 1e-5 * max|ref| (``mismatches``).  The backward replay starts from the kernel's own saved outputs and
loss cotangents, so a forward error does not leak into the backward's comparison.

The replay also recomputes what the kernel's controller saw, in float64:
  * the first dt of every solve (the forward's, and every backward interval's) equals Hairer's estimate from the
    replayed start state to 1e-4 (1e-3 under the seminorm, whose d2 carries the rounding of two fp32 RHS values h0
    apart: ``test_dopri5_seminorm_with_rejected_steps``), or the caller's ``first_step`` -- this catches a wrong norm of
    any block, theta's included;
  * at rtol 1e-5 / 1e-4, where the controller works above the noise floor: every dt after the first of a solve is
    dt * factor(ratio64) of the attempt before it to 2 % (where ratio64 >= 0.05; below it the ratio is fp32 noise of a
    nearly exact step), and every accept decision is ratio64 <= 1 unless |ratio64 - 1| < 5 %.

One replay with all six parameter cotangents serves every adjoint option: the y / adj_y algebra never reads theta, so S,
the seminorm and ``first_step`` change only the step sequence (which comes from the log) and the norm of the controller
checks (``adjoint_backward_t``'s).  The tensor-core streaming case (B >= 5: 3xTF32 contractions, DESIGN.md section 3.2)
is held to the same bar.

Observed on a B200 (1000 W power limit), maxima over the cases of relative L2 / element-wise error over max|ref|: y
7.9e-7 / 3.5e-6, adj_y0 1.6e-6 / 3.1e-6, gradients 2.1e-6 / 3.5e-6 (the tensor-core case; fp32 contractions 1.2e-6 /
2.9e-6), t.grad 4.1e-6 / 3.2e-6; every first dt within 1e-4, later dt within 1e-4 of dt * factor(ratio64) (92 checked).
On the parent of the fix of DESIGN.md section 8 the rows problems whose first backward interval took an even number of
accepted steps failed: first dt of the next interval 35-50 % off, Ws / Wp relative L2 up to 1.5e-4
(``profiles/r12a_replay*.txt``).  The whole file runs in about 2 minutes, most of it the float64 replays of the breast-shape and 16 000-gene cases.
"""
import collections

import pytest
import torch

import phoenix_b200 as pbm
from oracle import phoenix_oracle as O
from golden_util import rel_l2
from test_gpu_adjoint_params import _oracle_problem
from test_gpu_adjoint_seminorm import _problem
from test_gpu_placements import _set_knobs, make_net, mismatches
from test_gpu_time_grad import adjoint_backward_t

NAMES = O.PARAM_ORDER
F64 = torch.float64
TOL = 1e-5             # relative L2 and element-wise / max|ref|, every output
FIRST_RTOL = 1e-4      # first dt of a solve against the float64 Hairer estimate
CTRL_RTOL = 2e-2       # dt after the first against dt * factor(ratio64) of the attempt before
CTRL_RATIO_MIN = 0.05  # ... where ratio64 is at least this
DECIDE_BAND = 0.05     # accept decisions are checked where |ratio64 - 1| >= this


# ---- replay of the oracle's own logs (CPU) ----------------------------------------------------------------------------------
def _cpu_case(T, dtype=torch.float32):
    w, _, _, _ = _oracle_problem()
    gen = torch.Generator().manual_seed(70 + T)
    y0 = torch.rand(1, w.G, generator=gen)
    t = torch.linspace(0.0, 0.15 * (T - 1), T, dtype=F64)
    target = torch.rand(T - 1, 1, w.G, generator=gen)
    if dtype != torch.float32:
        w = O.Weights(*[p.to(dtype) for p in w.as_list()])
        y0, target = y0.to(dtype), target.to(dtype)
    y, flog = O.odeint(w, y0, t, method="dopri5")
    gy = torch.zeros_like(y)
    gy[1:] = 2.0 * (y[1:] - target)
    return w, y0, t, y, gy, flog


@pytest.mark.parametrize("T", [2, 3, 5])
def test_oracle_replaying_its_own_log_is_itself(T):
    """fp32: the replay of the oracle's own forward and backward logs is the oracle, bit for bit (outputs, steps, error
    ratios and initial-step estimates); the extension of test_gpu_time_grad replays the same way."""
    w, y0, t, y, gy, flog = _cpu_case(T)
    y2, flog2 = O.odeint(w, y0, t, method="dopri5", replay=flog.steps)
    assert torch.equal(y2, y)
    assert flog2.steps == flog.steps and flog2.ratios == flog.ratios and flog2.starts == flog.starts
    a, g, blog = O.adjoint_backward(w, t, y, gy, method="dopri5")
    assert len(blog.starts) == T - 1
    a2, g2, blog2 = O.adjoint_backward(w, t, y, gy, method="dopri5", replay=blog.steps)
    assert torch.equal(a2, a) and all(torch.equal(x, z) for x, z in zip(g2, g))
    assert blog2.steps == blog.steps and blog2.ratios == blog.ratios and blog2.starts == blog.starts
    a3, g3, blog3, _ = adjoint_backward_t(w, t, y, gy, replay=blog.steps)
    assert torch.equal(a3, a) and all(torch.equal(x, z) for x, z in zip(g3, g))
    assert blog3.ratios == blog.ratios


def test_float64_replay_of_a_float32_log_is_close():
    """The float64 replay of the fp32 oracle's logs differs from the fp32 run by its rounding only (<= 1e-6)."""
    w, y0, t, y, gy, flog = _cpu_case(3)
    a, g, blog = O.adjoint_backward(w, t, y, gy, method="dopri5")
    wd = O.Weights(*[p.double() for p in w.as_list()])
    y64, _ = O.odeint(wd, y0.double(), t, method="dopri5", replay=flog.steps)
    assert rel_l2(y, y64) <= 1e-6, rel_l2(y, y64)
    a64, g64, _ = O.adjoint_backward(wd, t, y.double(), gy.double(), method="dopri5", replay=blog.steps)
    assert rel_l2(a, a64) <= 1e-6, rel_l2(a, a64)
    for i in range(6):
        assert rel_l2(g[i], g64[i]) <= 1e-6, (NAMES[i], rel_l2(g[i], g64[i]))


def test_a_malformed_log_is_refused():
    w, y0, t, y, gy, flog = _cpu_case(3)
    _, _, blog = O.adjoint_backward(w, t, y, gy, method="dopri5")
    fwd, bwd = list(flog.steps), list(blog.steps)
    k = next(i for i, s in enumerate(fwd[:-1]) if s[2])   # an accepted attempt before the last
    assert len(blog.starts) == 2
    e = blog.starts[1][0] - 1                            # the last attempt of the first backward interval

    def fwd_with(steps):
        O.odeint(w, y0, t, method="dopri5", replay=steps)

    def bwd_with(steps):
        O.adjoint_backward(w, t, y, gy, method="dopri5", replay=steps)

    gap = fwd[:k + 1] + [(fwd[k + 1][0] + 1e-3 * fwd[k + 1][1],) + fwd[k + 1][1:]] + fwd[k + 2:]
    with pytest.raises(AssertionError, match="starts at"):
        fwd_with(gap)
    changed = fwd[:k] + [(fwd[k][0], fwd[k][1] * 1.01, True)] + fwd[k + 1:]
    with pytest.raises(AssertionError, match="starts at"):
        fwd_with(changed)
    with pytest.raises(AssertionError, match="ends at attempt"):
        fwd_with(fwd[:-1])
    with pytest.raises(AssertionError, match="left over"):
        fwd_with(fwd + [(fwd[-1][0] + fwd[-1][1], fwd[-1][1], True)])
    # an interval that ends short: the next interval's first attempt does not start where its last step ended
    with pytest.raises(AssertionError, match="starts at"):
        bwd_with(bwd[:e] + bwd[e + 1:])
    # ... or whose last step is not the one that covers its output time
    short = bwd[:e] + [(bwd[e][0], bwd[e][1] * 0.5, True)] + bwd[e + 1:]
    with pytest.raises(AssertionError, match="starts at"):
        bwd_with(short)
    bwd_with(bwd)


# ---- GPU ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pb():
    pbm.set_sync_errors(True)
    yield pbm
    pbm.set_step_logging(False)
    pbm.engine.FORCE_ENGINE = None


Case = collections.namedtuple("Case", "name engine G H shape many times rtol S semi first_step tgrad loss_all gmin rpp")
ALL = (0, 1, 2, 3, 4, 5)
T3 = (0.0, 0.1, 0.2)
T5 = (0.0, 0.1, 0.2, 0.3, 0.4)


def C(name, engine, G, H, shape, many, times, rtol=1e-7, S=ALL, semi=False, first_step=None, tgrad=False,
      loss_all=True, gmin=None, rpp=None):
    return Case(name, engine, G, H, shape, many, times, rtol, S, semi, first_step, tgrad, loss_all, gmin, rpp)


# rpp: rows per adjoint pass of the rows cases (the placement shapes of test_gpu_placements, DESIGN.md section 4)
CASES = [
    C("res-B1-T5", "resident", 350, 40, (1, 350), False, T5),
    C("res-B1-T2-semi", "resident", 350, 40, (1, 350), False, (0.0, 0.3), rtol=1e-5, semi=True),
    C("res-B3-T3-sub-last", "resident", 350, 40, (3, 1, 350), False, T3, rtol=1e-5, S=(5, 0), loss_all=False),
    C("res-B1-T3-first-tgrad", "resident", 350, 40, (1, 350), False, T3, rtol=1e-5, first_step=0.02, tgrad=True),
    C("rows4-T3", "rows", 690, 200, (5, 1, 690), True, T3, rpp=4),
    C("rows4-T5", "rows", 690, 200, (5, 1, 690), True, T5, rtol=1e-5, rpp=4),
    C("rows4-T3-last-tgrad", "rows", 690, 200, (5, 1, 690), True, T3, rtol=1e-5, loss_all=False, tgrad=True, rpp=4),
    C("rows4-T3-first", "rows", 690, 200, (5, 1, 690), True, T3, first_step=0.02, rpp=4),
    C("rows2-T3-semi", "rows", 13000, 129, (3, 1, 13000), True, T3, rtol=1e-5, semi=True, rpp=2),
    C("rows1-T3-sub", "rows", 16000, 100, (2, 1, 16000), True, T3, S=(0, 1, 3, 4), rpp=1),
    C("rows1-T3-reject", "rows", 1001, 100, (2, 1, 1001), True, (0.0, 2.0, 5.0), rtol=1e-4, gmin="110", rpp=1),
    C("rows-breast-T3", "rows", 11165, 200, (2, 1, 11165), True, T3, rpp=None),
    C("stream-B2-T3", "stream", 350, 40, (2, 350), False, T3, rtol=1e-5),
    C("stream-B6-T3-tc", "stream", 350, 40, (6, 350), False, T3),
]

# what the rows cases exercised, for test_rows_cases_cover_the_interval_parities
_SEEN = {}


def _gpu_run(pb, net, y0, t, target, c):
    """Forward + backward on the GPU with step logging.  Returns y, adj_y0, the six .grad (None outside S), t.grad (or
    None) and the forward and backward logs per problem."""
    plist = list(net.parameters())
    saved = pb.engine.FORCE_ENGINE
    pb.engine.FORCE_ENGINE = c.engine
    pb.set_step_logging(True)
    try:
        net.zero_grad(set_to_none=True)
        kw, opts = {}, {}
        if c.S != ALL:
            kw["adjoint_params"] = [plist[i] for i in c.S]
        if c.semi:
            opts["norm"] = "seminorm"
        if c.first_step is not None:
            opts["first_step"] = c.first_step
        if opts:
            kw["adjoint_options"] = opts
        y0g = y0.cuda().requires_grad_(True)
        tg = t.clone().requires_grad_(True) if c.tgrad else t
        n = y0.shape[0] if c.many else 1
        solve = pb.odeint_adjoint_many if c.many else pb.odeint_adjoint
        y = solve(net, y0g, tg, rtol=c.rtol, atol=c.rtol * 1e-2, method="dopri5", **kw)
        flogs = [pb.last_step_log(i) for i in range(n)] if c.many else [pb.last_step_log()]
        _loss(y, target.cuda(), c).backward()
        blogs = [pb.last_step_log(i) for i in range(n)] if c.many else [pb.last_step_log()]
        grads = [None if p.grad is None else p.grad.detach().cpu().clone() for p in plist]
        return y.detach().cpu(), y0g.grad.cpu(), grads, (tg.grad if c.tgrad else None), flogs, blogs
    finally:
        pb.set_step_logging(False)
        pb.engine.FORCE_ENGINE = saved


def _loss(y, target, c):
    """sum of squares on every output after the first, or on the last one only (y: [T, ...] or [N, T, ...])."""
    if c.many:
        return (((y[:, 1:] - target) if c.loss_all else (y[:, -1] - target[:, -1])) ** 2).sum()
    return (((y[1:] - target) if c.loss_all else (y[-1] - target[-1])) ** 2).sum()


def _cotangent(yk, tk, c):
    """The loss cotangent of one problem's outputs yk [T, ...] (float64) with targets tk [T-1, ...]."""
    gy = torch.zeros_like(yk)
    if c.loss_all:
        gy[1:] = 2.0 * (yk[1:] - tk)
    else:
        gy[-1] = 2.0 * (yk[-1] - tk[-1])
    return gy


def _controller(mine, log64, c, backward):
    """Where the kernel's log departs from what the float64 replay computes its controller should have done."""
    bad = []
    semi = backward and c.semi
    first = c.first_step if backward else None
    starts = set()
    for i, h in log64.starts:
        starts.add(i)
        want = first if first is not None else h
        tol = 1e-3 if semi else FIRST_RTOL
        if abs(mine[i][1] - want) > tol * abs(want):
            bad.append("first dt of the solve at attempt %d: %r, want %r (%.1e)" % (i, mine[i][1], want,
                                                                                  abs(mine[i][1] / want - 1)))
    if c.rtol < 1e-5:
        return bad, 0
    worst, n = 0.0, 0
    for k in range(1, len(mine)):
        r = log64.ratios[k - 1]
        if k in starts or not r >= CTRL_RATIO_MIN:
            continue
        want = float(O._next_dt(torch.tensor(mine[k - 1][1], dtype=F64), torch.tensor(r, dtype=F64)))
        dev = abs(mine[k][1] / want - 1)
        worst, n = max(worst, dev), n + 1
        if dev > CTRL_RTOL:
            bad.append("dt of attempt %d: %r, want %r from ratio64 %.4f (%.1e)" % (k, mine[k][1], want, r, dev))
    for k, (s, r) in enumerate(zip(mine, log64.ratios)):
        if abs(r - 1) >= DECIDE_BAND and bool(s[2]) != (r <= 1):
            bad.append("attempt %d %s at ratio64 %.4f" % (k, "accepted" if s[2] else "rejected", r))
    print("    controller: %d dt checked, worst %.1e" % (n, worst))
    return bad, n


def _accepted_per_interval(log64):
    """Accepted steps of each solve of a replay log (the backward's: one per interval, T-1 first)."""
    bounds = [i for i, _ in log64.starts] + [len(log64.steps)]
    return [sum(1 for s in log64.steps[a:b] if s[2]) for a, b in zip(bounds, bounds[1:])]


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=[c.name for c in CASES])
def test_dopri5_against_float64_replay(pb, monkeypatch, c):
    _set_knobs(monkeypatch, pb, c.gmin)
    w, y0, t, target = _problem(c.G, c.H, c.shape, c.many, c.times, 900 + c.G % 97 + 7 * len(c.times))
    net = make_net(pb, w)
    y, ady, grads, tgrad, flogs, blogs = _gpu_run(pb, net, y0, t, target, c)
    wd = O.Weights(*[p.double() for p in w.as_list()])
    probs = range(y0.shape[0]) if c.many else [None]
    y64, a64, g64, tv64, bad, counts = [], [], None, [], [], []
    print("\n%s (%s, %d x %d, y0 %s, T = %d, rtol %.0e)" % (c.name, c.engine, c.G, c.H, tuple(c.shape), len(c.times),
                                                               c.rtol))
    for k in probs:
        pick = (lambda x: x[k]) if c.many else (lambda x: x)
        i = 0 if k is None else k
        yk, flog64 = O.odeint(wd, pick(y0).double(), pick(t), method="dopri5", rtol=c.rtol, atol=c.rtol * 1e-2,
                              replay=flogs[i])
        yker = pick(y).double()
        ak, gk, blog64, tvk = adjoint_backward_t(wd, pick(t), yker, _cotangent(yker, pick(target).double(), c),
                                                 "dopri5", c.rtol, c.rtol * 1e-2, t_requires_grad=c.tgrad,
                                                 semi=c.semi, params=c.S, replay=blogs[i])
        y64.append(yk)
        a64.append(ak)
        tv64.append(tvk)
        g64 = gk if g64 is None else [a + b for a, b in zip(g64, gk)]
        acc = _accepted_per_interval(blog64)
        counts.append((acc, len(blogs[i])))
        print("  problem %d: forward %d attempts, backward %d attempts, accepted per interval (T-1 .. 1) %s"
              % (i, len(flogs[i]), len(blogs[i]), acc))
        for what, mine, log64, backward in (("fwd", flogs[i], flog64, False), ("bwd", blogs[i], blog64, True)):
            msgs, _ = _controller(mine, log64, c, backward)
            bad += ["problem %d %s: %s" % (i, what, m) for m in msgs]
    st = torch.stack if c.many else (lambda v: v[0])
    y64, a64 = st(y64), st(a64)
    bad += mismatches("y", y, y64, TOL)
    bad += mismatches("adj_y0", ady, a64, TOL)
    for i in range(6):
        if i in c.S:
            bad += mismatches(NAMES[i], grads[i], g64[i], TOL)
        elif grads[i] is not None and bool(grads[i].any()):
            bad.append("%s is outside the adjoint set and has a gradient" % NAMES[i])
    if c.tgrad:
        bad += mismatches("t.grad", tgrad, st(tv64), TOL)
    if c.engine == "rows":
        _SEEN[c.name] = (counts, c.rpp, any(not s[2] for lg in blogs + flogs for s in lg))
    print("  " + ("FAILED:\n    " + "\n    ".join(bad) if bad else "ok"))
    assert not bad, "\n".join(bad)


@pytest.mark.gpu
def test_rows_cases_cover_the_interval_parities():
    """The rows cases exercise what the rows adjoint's per-interval state handling depends on: some backward interval
    after the first follows one with an even number of accepted steps and some one with an odd number (the FSAL slot
    swaps leave the slot maps in the other state), at least one attempt is rejected, and the rows of one pass take
    different numbers of attempts."""
    rows = [c.name for c in CASES if c.engine == "rows"]
    missing = [n for n in rows if n not in _SEEN]
    if missing:
        pytest.skip("needs the rows cases of test_dopri5_against_float64_replay in the same run: %s" % missing)
    parities, rejects, uneven = set(), False, False
    for name in rows:
        counts, rpp, rej = _SEEN[name]
        rejects |= rej
        for acc, _ in counts:
            parities |= {n % 2 for n in acc[:-1]}   # intervals followed by another one
        if rpp and rpp > 1:
            for lo in range(0, len(counts), rpp):
                uneven |= len({n for _, n in counts[lo:lo + rpp]}) > 1
    assert parities == {0, 1}, parities
    assert rejects, "no rows case rejects an attempt"
    assert uneven, "the rows of every pass take the same number of backward attempts"


@pytest.mark.gpu
def test_resident_many_is_the_replayed_single_call(pb):
    """odeint_adjoint_many on the resident engine runs several problems per launch and logs no steps.  Each problem's y
    and adj_y0 equal the single-problem call's bit for bit, and the gradients the sum of the single calls' (in the order
    the many call sums them); the single calls are held to the float64 replay of their own logs."""
    c = C("res-many", "resident", 350, 40, (3, 1, 350), True, T3, rtol=1e-5)
    w, y0, t, target = _problem(c.G, c.H, c.shape, True, c.times, 77)
    net = make_net(pb, w)
    plist = list(net.parameters())
    saved = pb.engine.FORCE_ENGINE
    pb.engine.FORCE_ENGINE = "resident"
    try:
        net.zero_grad(set_to_none=True)
        y0g = y0.cuda().requires_grad_(True)
        y = pb.odeint_adjoint_many(net, y0g, t, rtol=c.rtol, atol=c.rtol * 1e-2, method="dopri5")
        _loss(y, target.cuda(), c).backward()
        many = (y.detach().cpu(), y0g.grad.cpu(), [p.grad.clone() for p in plist])
    finally:
        pb.engine.FORCE_ENGINE = saved
    one = C("res-one", "resident", 350, 40, (1, 350), False, T3, rtol=c.rtol)
    ys, adys, gs, bad = [], [], [], []
    wd = O.Weights(*[p.double() for p in w.as_list()])
    for k in range(3):
        yk, ak, gk, _, flogs, blogs = _gpu_run(pb, net, y0[k], t[k], target[k], one)
        ys.append(yk)
        adys.append(ak)
        gs.append(gk)
        y64, _ = O.odeint(wd, y0[k].double(), t[k], method="dopri5", rtol=c.rtol, atol=c.rtol * 1e-2, replay=flogs[0])
        a64, g64, _, _ = adjoint_backward_t(wd, t[k], yk.double(), _cotangent(yk.double(), target[k].double(), one),
                                            "dopri5", c.rtol, c.rtol * 1e-2, replay=blogs[0])
        bad += mismatches("y", yk, y64, TOL) + mismatches("adj_y0", ak, a64, TOL)
        bad += sum((mismatches(NAMES[i], gk[i], g64[i], TOL) for i in range(6)), [])
    assert not bad, "\n".join(bad)
    assert torch.equal(many[0], torch.stack(ys))
    assert torch.equal(many[1], torch.stack(adys))
    for i in range(6):
        ref = torch.stack([g[i].cuda() for g in gs]).sum(dim=0)
        assert torch.equal(many[2][i], ref), (NAMES[i], rel_l2(many[2][i].cpu(), ref.cpu()))
