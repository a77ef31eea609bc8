"""Every on-chip weight placement of the resident and rows solver kernels against a float64 oracle.

For every call the host planners (``phx_resident_plan`` / ``phx_rows_plan``, csrc/phx_plan.cu) decide where a CTA's two
weight slices live -- resident in shared memory, WA parked in tensor memory, or streamed from L2 through a per-warp ring
of 1..4 TMA slots that doubles as the cross-warp reduction buffer -- and which kernel template runs (NV = 1 / 2 / 4
float4 columns per lane, batch blocks of PassRows<NV, BT> rows, quad-warp layouts of the rows kernels, 1 / 2 / 4 rows
per adjoint pass).  A stale ring slot or a wrong parity bit gives plausible numbers from the wrong weight row, so each
tier is run here at a shape the planner sends to it and compared with a float64 solve of the oracle.

The class of a call is
  * resident: (NV, w1, wa, min(ring_stages, 2)) with w1 / wa = 1 shared memory, 2 tensor memory, 0 streamed;
  * rows:     (nqw, wa, rows per pass).
``CASES`` holds one or more calls per class; ``test_table_covers_every_planner_class`` (no GPU) checks that every class
the planners produce over G in [37, 30 000], H in [1, 256], B in 1..8 forward / 1..4 adjoint is in the table, and that
every case still lands on its class at 148 SMs.

Tolerances (fixed grid), with the maxima observed over every case on a B200 (148 SMs, 1000 W power limit) in brackets:
  * relative L2 <= 1e-5 for y, adj_y0 and the six parameter gradients [y 2.1e-8, adj_y0 7.4e-8, gradients 1.4e-7];
  * element-wise max|a - r| <= c * max|r| per tensor, c = 1e-5 [y 1.1e-7, adj_y0 1.9e-7, gradients 3.0e-7].
    Relative L2 over 20 000 genes absorbs one gene off by 1e-3; this bound does not: one WA row scaled by 1 + 1e-3 moves
    y by 1.7e-4 (WA in tensor memory, 11 165 genes) and 6.7e-5 (WA ring, 20 000 genes) of max|y| while relative L2 stays
    at 1.8e-6 / 5.5e-7 (``test_one_wrong_weight_row_is_rejected``).
Weights above 1 000 genes are scaled (``_inputs``) so that every case integrates well-conditioned dynamics.
"""
import ctypes
import collections

import pytest
import torch

from golden_util import assert_logs_close, compare_logs, rel_l2
from oracle import phoenix_oracle as O

SMS = 148
C_STATE, C_GRAD, L2_TOL = 1e-5, 1e-5, 1e-5

Case = collections.namedtuple("Case", "kernel adjoint G H n method cls stages")


def R(adjoint, G, H, B, cls, stages=0, method="rk4"):
    """Resident call on a batch of B rows (y0 of shape (B, 1, G)); cls = (NV, w1, wa, min(S, 2)), stages = exact S."""
    return Case("resident", adjoint, G, H, B, method, cls, stages)


def W(adjoint, G, H, N, cls, method="rk4"):
    """Rows call of odeint_adjoint_many on N one-row problems; cls = (nqw, wa, rows per pass)."""
    return Case("rows", adjoint, G, H, N, method, cls, None)


F, A = 0, 1
# PassRows blocks (BT = 4 for B > 1): NV 1 -> 4 fwd / 4 adj, NV 2 -> 4 / 2, NV 4 -> 2 / 1.  B = 3, 5, 6, 7 leave a ragged
# last block for every (NV, direction) whose block exceeds one row.
CASES = [
    # ---- resident forward
    R(F, 350, 40, 7, (1, 1, 1, 0)),                        # NV 1, both slices in shared memory, ragged block (4 + 3)
    R(F, 24000, 64, 7, (1, 1, 2, 0), method="midpoint"),   # NV 1, WA in tensor memory, ragged block
    R(F, 3551, 120, 7, (2, 1, 1, 0)),                      # NV 2, both in shared memory, ragged block
    R(F, 24000, 65, 6, (2, 1, 2, 0)),                      # NV 2, WA in tensor memory, ragged block (4 + 2)
    R(F, 24000, 120, 7, (2, 0, 2, 2), 4),                  # NV 2, W1 ring (4 slots), WA in tensor memory
    R(F, 690, 160, 3, (4, 1, 1, 0)),                       # NV 4, both in shared memory, ragged block (2 + 1)
    R(F, 11165, 200, 4, (4, 1, 2, 0)),                     # breast shape, batch blocks
    R(F, 11165, 200, 8, (4, 1, 2, 0), method="euler"),
    R(F, 16000, 200, 7, (4, 0, 2, 2), 4),                  # NV 4, W1 ring, WA in tensor memory, ragged block
    R(F, 20000, 129, 1, (4, 1, 0, 2), 4),                  # WA ring at every depth; the fused pass walks 1..4 blocks
    R(F, 20000, 129, 3, (4, 1, 0, 2), 3),
    R(F, 20000, 129, 5, (4, 1, 0, 2), 2),
    R(F, 20000, 129, 7, (4, 1, 0, 1), 1),
    R(F, 20000, 200, 1, (4, 0, 0, 2), 4),                  # C5 shape: both slices streamed
    # ---- resident adjoint
    R(A, 350, 40, 3, (1, 1, 1, 0)),                        # NV 1, both in shared memory, one ragged block (3 of 4)
    R(A, 24000, 33, 3, (1, 1, 2, 0)),                      # NV 1, WA in tensor memory
    R(A, 30000, 33, 3, (1, 0, 2, 2), 4, method="euler"),   # NV 1, W1 ring
    R(A, 3551, 120, 3, (2, 1, 1, 0)),                      # NV 2, both in shared memory, ragged block (2 + 1)
    R(A, 8000, 128, 3, (2, 1, 2, 0)),                      # NV 2, WA in tensor memory, ragged block
    R(A, 24000, 120, 4, (2, 0, 2, 1), 1),                  # NV 2, W1 ring, 1 slot
    R(A, 20000, 128, 4, (2, 0, 2, 2), 2),                  # NV 2, W1 ring, 2 slots
    R(A, 690, 160, 3, (4, 1, 1, 0)),                       # NV 4, both in shared memory
    R(A, 37, 256, 3, (4, 1, 2, 0)),                        # H = 256 (K2q = 128: no padded lanes), WA in tensor memory
    R(A, 11165, 200, 1, (4, 1, 2, 0)),
    R(A, 350, 256, 4, (4, 0, 2, 1), 1),                    # W1 ring at every depth, WA in tensor memory
    R(A, 350, 256, 3, (4, 0, 2, 2), 2),
    R(A, 8000, 200, 3, (4, 0, 2, 2), 3),
    R(A, 11165, 200, 2, (4, 0, 2, 2), 3),
    R(A, 11165, 200, 4, (4, 0, 2, 2), 2),
    R(A, 20000, 129, 1, (4, 1, 0, 1), 1),                  # WA ring, 1 slot
    R(A, 19050, 129, 1, (4, 1, 0, 2), 2),                  # WA ring, 2 slots
    R(A, 20000, 200, 2, (4, 0, 0, 1), 1),                  # both streamed, 1 slot
    R(A, 20000, 129, 2, (4, 0, 0, 2), 4, method="midpoint"),
    R(A, 20000, 200, 1, (4, 0, 0, 2), 4),                  # C5 shape
    # ---- rows kernels (N problems; the forward always runs 4 rows per pass)
    W(F, 350, 40, 5, (1, 1, 4)),
    W(F, 1001, 100, 5, (2, 1, 4)),
    W(F, 690, 200, 5, (4, 1, 4)),                          # nqw 4, WA in shared memory
    W(F, 2049, 129, 5, (4, 1, 4)),                         # H = 129: NV "3" rounded up to 4, the most padding
    W(F, 11165, 160, 5, (4, 2, 4)),                        # nqw 4, WA in tensor memory
    W(A, 350, 40, 5, (1, 1, 4)),
    W(A, 1001, 100, 5, (2, 1, 4)),
    W(A, 690, 200, 5, (4, 1, 4)),
    W(A, 1001, 256, 5, (4, 1, 4), method="euler"),         # H = 256
    W(A, 2049, 129, 5, (4, 1, 4)),
    W(A, 11165, 160, 5, (4, 2, 4)),
    W(A, 13000, 129, 3, (4, 2, 2), method="midpoint"),     # 2 rows per adjoint pass (2 + 1)
    W(A, 16000, 100, 3, (4, 2, 1)),                        # 1 row per adjoint pass
]


def _case_id(c):
    return "%s-%s-%dx%d-%s%d-%s" % (c.kernel[:3], "adj" if c.adjoint else "fwd", c.G, c.H,
                                    "B" if c.kernel == "resident" else "N", c.n, c.method)


# ---- planner classes (host only) -------------------------------------------------------------------------------------------
def _lib():
    from phoenix_b200 import _lib as L
    return L.load()


def resident_plan(lib, sms, G, H, B, adjoint):
    """(class, ring_stages, nCTA, gpc) of the resident planner, or None when it refuses the shape."""
    out = (ctypes.c_int32 * 8)()
    if lib.phx_plan_describe(sms, G, H, B, adjoint, out) != 0:
        return None
    return (out[2], out[3], out[4], min(out[6], 2)), out[6], out[0], out[1]


def rows_plan(lib, sms, G, H, adjoint):
    """(class, nCTA, gpc) of the rows planner, or None when it refuses the shape."""
    out = (ctypes.c_int32 * 10)()
    if lib.phx_rows_plan_describe(sms, G, H, adjoint, out) != 0:
        return None
    return (out[2], out[5], out[6]), out[0], out[1]


def _tier_problem(lib, sms, c):
    """None if case c lands on its expected class (and ring depth) at `sms` SMs, else a description of where it went."""
    if c.kernel == "resident":
        got = resident_plan(lib, sms, c.G, c.H, c.n, c.adjoint)
        if got is not None and got[0] == c.cls and got[1] == c.stages:
            return None
        want = (c.cls, c.stages)
        got = None if got is None else got[:2]
    else:
        got = rows_plan(lib, sms, c.G, c.H, c.adjoint)
        if got is not None and got[0] == c.cls:
            return None
        want, got = c.cls, None if got is None else got[0]
    return "%s: expected (class, stages) %s at %d SMs, the planner gives %s" % (_case_id(c), want, sms, got)


GRID_G = (37, 129, 350, 690, 1001, 2048, 2049, 3551, 8000, 11165, 13000, 16000, 19050, 20000, 24000, 30000)
GRID_H = (1, 5, 33, 40, 64, 65, 100, 120, 128, 129, 130, 160, 192, 200, 256)


def test_table_covers_every_planner_class(monkeypatch):
    """No GPU needed: every case lands on its class at 148 SMs, and every class the planners produce over the grid has
    a case in the table (a planner change that creates a tier or moves a case fails here, not silently on the GPU)."""
    monkeypatch.delenv("PHX_NO_TMEM", raising=False)
    monkeypatch.delenv("PHX_MIN_GENES_PER_CTA", raising=False)
    monkeypatch.delenv("PHX_NO_ROWS", raising=False)
    lib = _lib()
    problems = [m for m in (_tier_problem(lib, SMS, c) for c in CASES) if m]
    assert not problems, "\n".join(problems)
    table = {(c.kernel, c.adjoint, c.cls) for c in CASES}
    seen = {}
    for adjoint in (0, 1):
        for G in GRID_G:
            for H in GRID_H:
                p = rows_plan(lib, SMS, G, H, adjoint)
                if p is not None:
                    seen.setdefault(("rows", adjoint, p[0]), (G, H))
                for B in range(1, (4 if adjoint else 8) + 1):
                    p = resident_plan(lib, SMS, G, H, B, adjoint)
                    if p is not None:
                        seen.setdefault(("resident", adjoint, p[0]), (G, H, B))
    missing = {k: v for k, v in seen.items() if k not in table}
    assert not missing, "planner classes without a case in CASES (class: first shape): %s" % missing
    # every ring depth 1..4 of both streamed slices, forward and adjoint, and ragged blocks for every NV
    for adjoint in (0, 1):
        for w1, wa in ((0, 2), (1, 0), (0, 0)):
            assert any(c.kernel == "resident" and c.adjoint == adjoint and c.cls[1:3] == (w1, wa) for c in CASES)
    assert {c.stages for c in CASES if c.kernel == "resident"} >= {1, 2, 3, 4}
    block = {(1, 0): 4, (1, 1): 4, (2, 0): 4, (2, 1): 2, (4, 0): 2, (4, 1): 1}
    for (nv, adjoint), pb in block.items():
        if pb > 1:
            assert any(c.kernel == "resident" and c.cls[0] == nv and c.adjoint == adjoint and c.n > 1 and c.n % pb
                       for c in CASES), (nv, adjoint)


# ---- GPU ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pb():
    import phoenix_b200 as pb
    pb.set_sync_errors(True)
    yield pb
    pb.set_step_logging(False)
    pb.engine.FORCE_ENGINE = None


def _num_sms():
    from phoenix_b200 import _lib as L
    return L.load().phx_ctx_num_sms(L.ctx(torch.cuda.current_device()))


def make_net(pb, w):
    net = pb.ODENet("cuda", w.G, neurons=w.H)
    with torch.no_grad():
        for p, src in zip(net.parameters(), w.as_list()):
            p.copy_(src)
    return net


def _inputs(c, seed, times=(0.0, 0.04, 0.1)):
    """Dense weights (a wrong row and the relu mask both matter), y0, output times (float64; each rows problem shifted
    by its own offset), loss target.  Above 1 000 genes the two input matrices are scaled by sqrt(1000 / G): the
    branch sums then stay O(1) as G grows (unscaled, exp of the prods branch reaches 1e3 at 24 000 genes and the state
    leaves [0, 1] and overflows within 0.1 time units)."""
    w = O.make_weights(c.G, c.H, seed, dense=True, neg_mult_frac=0.2)
    if c.G > 1000:
        w.Wp.mul_((1000.0 / c.G) ** 0.5)
        w.Ws.mul_((1000.0 / c.G) ** 0.5)
    gen = torch.Generator().manual_seed(seed + 1)
    if c.kernel == "resident":
        shape = (1, c.G) if c.n == 1 else (c.n, 1, c.G)
        t = torch.tensor(times, dtype=torch.float64)
        target = torch.rand(len(times) - 1, *shape, generator=gen)
    else:
        shape = (c.n, 1, c.G)
        tau = torch.rand(c.n, 1, generator=gen, dtype=torch.float64)
        t = tau + torch.tensor(times, dtype=torch.float64)
        target = torch.rand(c.n, len(times) - 1, 1, c.G, generator=gen)
    y0 = torch.rand(*shape, generator=gen)
    return w, y0, t, target


def _reference(w, y0, t, target, method, adjoint, kernel, dtype=torch.float64, rtol=1e-7, atol=1e-9):
    """The oracle in `dtype`: resident batches as one (B, 1, G) state (RMS norm over the batch, misc.py:10-11); rows
    problems one at a time with the parameter gradients summed.  Returns y, adj_y0, grads, [(flog, blog)]."""
    wd = O.Weights(*[p.to(dtype) for p in w.as_list()])
    probs = [(y0, t, target)] if kernel == "resident" else [(y0[i], t[i], target[i]) for i in range(y0.shape[0])]
    ys, adys, gsum, logs = [], [], None, []
    for y0i, ti, tgi in probs:
        y, flog = O.odeint(wd, y0i.to(dtype), ti.double(), method=method, rtol=rtol, atol=atol)
        ys.append(y)
        if not adjoint:
            logs.append((flog, None))
            continue
        gy = torch.zeros_like(y)
        gy[1:] = 2.0 * (y[1:] - tgi.to(dtype)) / target.numel()
        ady, grads, blog = O.adjoint_backward(wd, ti.double(), y, gy, method=method, rtol=rtol, atol=atol)
        adys.append(ady)
        gsum = grads if gsum is None else [a + b for a, b in zip(gsum, grads)]
        logs.append((flog, blog))
    if kernel == "resident":
        return ys[0], (adys[0] if adjoint else None), gsum, logs
    return torch.stack(ys), (torch.stack(adys) if adjoint else None), gsum, logs


def _run(pb, c, net, y0, t, target, rtol=1e-7, atol=1e-9):
    """The kernel under test on the GPU: y, adj_y0, grads (None for a forward case) and the step logs."""
    saved = pb.engine.FORCE_ENGINE
    pb.engine.FORCE_ENGINE = c.kernel if c.kernel == "resident" else "rows"
    try:
        net.zero_grad()
        y0g = y0.cuda().requires_grad_(bool(c.adjoint))
        if c.kernel == "resident":
            if c.adjoint:
                y = pb.odeint_adjoint(net, y0g, t, rtol=rtol, atol=atol, method=c.method)
            else:
                with torch.no_grad():
                    y = pb.odeint(net, y0g, t, rtol=rtol, atol=atol, method=c.method)
            flogs = [pb.last_step_log()]
        else:
            if c.adjoint:
                y = pb.odeint_adjoint_many(net, y0g, t, rtol=rtol, atol=atol, method=c.method)
            else:
                with torch.no_grad():
                    y = pb.odeint_adjoint_many(net, y0g, t, rtol=rtol, atol=atol, method=c.method)
            flogs = [pb.last_step_log(i) for i in range(c.n)]
        blogs = None
        if c.adjoint:
            loss = torch.mean(((y[:, 1:] if c.kernel == "rows" else y[1:]) - target.cuda()) ** 2)
            loss.backward()
            blogs = [pb.last_step_log()] if c.kernel == "resident" else [pb.last_step_log(i) for i in range(c.n)]
            return (y.detach().cpu(), y0g.grad.cpu(), [p.grad.detach().cpu() for p in net.parameters()],
                    flogs, blogs)
        return y.cpu(), None, None, flogs, blogs
    finally:
        pb.engine.FORCE_ENGINE = saved


def mismatches(name, a, r, c, l2=L2_TOL):
    """Why `a` (fp32 kernel result) is not close enough to `r` (reference): relative L2 above `l2`, or an element
    further than c * max|r| from its reference value.  Empty when it is close."""
    a, r = a.double().reshape(-1), r.double().reshape(-1)
    rel = rel_l2(a, r)
    scale = float(r.abs().max())
    emax = float((a - r).abs().max())
    ratio = emax / scale if scale > 0 else emax
    print("%-8s rel_l2 %.2e  max|a-r|/max|r| %.2e" % (name, rel, ratio))
    out = []
    if not rel <= l2:
        out.append("%s: relative L2 %.3e > %.0e" % (name, rel, l2))
    if not ratio <= c:
        i = int((a - r).abs().argmax())
        out.append("%s: element %d off by %.3e (%.3e of max|ref|) > %.0e" % (name, i, float(a[i] - r[i]), ratio, c))
    return out


def _all_mismatches(y, ady, grads, y_ref, ady_ref, g_ref):
    bad = mismatches("y", y, y_ref, C_STATE)
    if ady is not None:
        bad += mismatches("adj_y0", ady, ady_ref, C_STATE)
        for i, (g, r) in enumerate(zip(grads, g_ref)):
            bad += mismatches("grad%d" % i, g, r, C_GRAD)
    return bad


def _check_tier(c):
    sms = _num_sms()
    msg = _tier_problem(_lib(), sms, c)
    assert msg is None, msg + " (the device has %d SMs; the table is laid out for %d)" % (sms, SMS)


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=[_case_id(c) for c in CASES])
def test_placement_against_fp64(pb, c):
    _check_tier(c)
    w, y0, t, target = _inputs(c, 6000 + c.G % 997 + 7 * c.H + 31 * c.n + c.adjoint)
    y, ady, grads, _, _ = _run(pb, c, make_net(pb, w), y0, t, target)
    y_ref, ady_ref, g_ref, _ = _reference(w, y0, t, target, c.method, c.adjoint, c.kernel)
    moved = rel_l2(y[:, -1] if c.kernel == "rows" else y[-1], y0)
    assert moved > 1e-3, "the state barely moved (%.2e): the case tests nothing" % moved
    bad = _all_mismatches(y, ady, grads, y_ref, ady_ref, g_ref)
    assert not bad, "\n".join(bad)


# ---- dopri5 on the ring tiers: the controller, rejected steps and ring_drain / redo ------------------------------------------
# (adjoint case, PHX_MIN_GENES_PER_CTA, output times).  Raising the genes per CTA sends a 1 001-gene model to the streamed
# tiers, so the ring code runs at a size whose tight-tolerance float64 solve is cheap.  Over these intervals the oracle's
# backward sweeps reject 1..3 attempts.
DOPRI = [
    (R(A, 350, 256, 3, (4, 0, 2, 2), 2, method="dopri5"), None, (0.0, 2.0, 5.0)),          # W1 ring
    (R(A, 1001, 129, 1, (4, 1, 0, 1), 1, method="dopri5"), "136", (0.0, 2.0, 5.0)),       # WA ring
    (R(A, 1001, 200, 1, (4, 0, 0, 2), 4, method="dopri5"), "200", (0.0, 2.0, 5.0)),       # both streamed
    (W(A, 1001, 100, 2, (4, 2, 1), method="dopri5"), "110", (0.0, 2.0, 5.0)),              # rows, 1 row per pass
]


def _set_knobs(monkeypatch, pb, gmin=None, no_tmem=False):
    """Planner knobs for one test (the planner reads them on every call); the engine's cache of rows-per-pass answers is
    reset with them."""
    if gmin is None:
        monkeypatch.delenv("PHX_MIN_GENES_PER_CTA", raising=False)
    else:
        monkeypatch.setenv("PHX_MIN_GENES_PER_CTA", str(gmin))
    if no_tmem:
        monkeypatch.setenv("PHX_NO_TMEM", "1")
    else:
        monkeypatch.delenv("PHX_NO_TMEM", raising=False)
    monkeypatch.setattr(pb.engine, "_rows_cache", {})


@pytest.mark.gpu
@pytest.mark.parametrize("c,gmin,times", DOPRI, ids=["%s-gmin%s" % (_case_id(c), g) for c, g, _ in DOPRI])
def test_dopri5_ring_tiers(pb, monkeypatch, c, gmin, times):
    """Loose tolerances (rtol 1e-4, atol 1e-6), where the controller works above the fp32 noise floor (DESIGN.md 5): the
    step logs follow the fp32 oracle's to 2 % (0.25 for a log whose step sequence the oracle itself does not reproduce in
    float64), the kernel rejects an attempt where the oracle does (a rejection redoes the step: the ring is drained and
    refilled for the retry), and y and the gradients are no further from a float64
    solve at rtol 1e-8 than 3x the fp32 oracle's own distance (the rule of test_dopri5_accuracy_against_fp64_truth; the
    float64 solve is 100x closer to the exact solution than the fp32 one at rtol 1e-4)."""
    _set_knobs(monkeypatch, pb, gmin)
    _check_tier(c)
    rtol, atol = 1e-4, 1e-6
    w, y0, t, target = _inputs(c, 5100 + c.H, times)
    pb.set_step_logging(True)
    try:
        y, ady, grads, flogs, blogs = _run(pb, c, make_net(pb, w), y0, t, target, rtol=rtol, atol=atol)
    finally:
        pb.set_step_logging(False)
    y32, ady32, g32, logs = _reference(w, y0, t, target, "dopri5", True, c.kernel, torch.float32, rtol, atol)
    _, _, _, logs64 = _reference(w, y0, t, target, "dopri5", True, c.kernel, torch.float64, rtol, atol)
    y64, ady64, g64, _ = _reference(w, y0, t, target, "dopri5", True, c.kernel, torch.float64, 1e-8, 1e-10)
    mine_all = []
    for i, (pair32, pair64) in enumerate(zip(logs, logs64)):
        for mine, ref, ref64, what in ((flogs[i], pair32[0].steps, pair64[0].steps, "fwd %d" % i),
                                       (blogs[i], pair32[1].steps, pair64[1].steps, "bwd %d" % i)):
            # 2 % where the oracle's own float32 and float64 step sequences agree to 2 % (the controller works above
            # the rounding noise); otherwise the noise-floor rule (0.25).  The first step of a backward sweep starts
            # from zero parameter cotangents and an error ratio far below 1, so the step after it is noise-decided.
            above = compare_logs(ref, ref64, 2e-2)[1] == "identical"
            assert_logs_close(mine, ref, 2e-2 if above else 0.25, what)
            mine_all += mine
    assert any(not s[2] for pair in logs for log in pair for s in log.steps), "the oracle rejects no step"
    assert any(not s[2] for s in mine_all), "the oracle rejects a step, the kernel never does"
    assert rel_l2(y, y64) <= 3 * rel_l2(y32, y64) + 2e-7
    assert rel_l2(ady, ady64) <= 3 * rel_l2(ady32, ady64) + 5e-6
    for i, (g, r32, r64) in enumerate(zip(grads, g32, g64)):
        assert rel_l2(g, r64) <= 3 * rel_l2(r32, r64) + 5e-6, (i, rel_l2(g, r64), rel_l2(r32, r64))


@pytest.mark.gpu
@pytest.mark.parametrize("gmin,cls,stages", [("128", (4, 0, 2, 2), 4), ("200", (4, 0, 0, 2), 4)])
def test_min_genes_per_cta_ring_tiers_rk4(pb, monkeypatch, gmin, cls, stages):
    """1 001 x 200, B = 1: 128 genes per CTA send the adjoint to a W1 ring with WA in tensor memory, 200 stream both
    slices.  nCTA changes with the knob, so the comparison is with the float64 oracle, not bit for bit."""
    _set_knobs(monkeypatch, pb, gmin)
    c = R(A, 1001, 200, 1, cls, stages)
    _check_tier(c)
    w, y0, t, target = _inputs(c, 5300)
    y, ady, grads, _, _ = _run(pb, c, make_net(pb, w), y0, t, target)
    y_ref, ady_ref, g_ref, _ = _reference(w, y0, t, target, "rk4", True, "resident")
    bad = _all_mismatches(y, ady, grads, y_ref, ady_ref, g_ref)
    assert not bad, "\n".join(bad)


# ---- placement invariance: WA in tensor memory or streamed through the ring, same bits ---------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("method", ["rk4", "dopri5"])
def test_wa_in_tensor_memory_or_ring_gives_identical_bits(pb, monkeypatch, method):
    """PHX_NO_TMEM moves WA from tensor memory to the ring at the same G, H, B (same nCTA / gpc): at 11 165 x 200, B = 1,
    the forward goes to a 3-slot WA ring and the adjoint to a 2-slot one.  With W1 resident the fused passes run the same
    row_fn / group_fn on the same rows in the same order -- only where a row is read from changes -- so y, adj_y0 and all
    six gradients must be equal bit for bit."""
    G, H = 11165, 200
    c = R(A, G, H, 1, (4, 1, 2, 0), method=method)
    w, y0, t, target = _inputs(c, 5400)
    net = make_net(pb, w)
    lib, sms = _lib(), _num_sms()
    out = {}
    for no_tmem in (False, True):
        _set_knobs(monkeypatch, pb, None, no_tmem)
        plans = [resident_plan(lib, sms, G, H, 1, adj) for adj in (0, 1)]
        if no_tmem:
            assert [p[0][:3] for p in plans] == [(4, 1, 0), (4, 1, 0)] and all(p[1] >= 1 for p in plans), plans
        else:
            assert [p[0] for p in plans] == [(4, 1, 2, 0), (4, 1, 2, 0)], plans
        out[no_tmem] = ([p[2:] for p in plans], _run(pb, c, net, y0, t, target)[:3])
    assert out[False][0] == out[True][0], "nCTA / gpc changed with PHX_NO_TMEM"
    a, b = out[False][1], out[True][1]
    assert torch.equal(a[0], b[0]), "y"
    assert torch.equal(a[1], b[1]), "adj_y0"
    for i, (ga, gb) in enumerate(zip(a[2], b[2])):
        assert torch.equal(ga, gb), "grad%d" % i


# ---- negative control: the bounds see one wrong weight row --------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("c", [R(F, 11165, 200, 1, (4, 1, 2, 0)), R(F, 20000, 129, 1, (4, 1, 0, 2), 4)],
                         ids=["wa-tensor-memory", "wa-ring"])
def test_one_wrong_weight_row_is_rejected(pb, c):
    """The kernel gets WA with one row scaled by 1 + 1e-3, the oracle the unmodified weights: the comparison must reject
    the result.  The row is a gene of the last warp of the last CTA (warp w owns rows w, w + 16, ... of its CTA's slice):
    of that warp's rows the one with the largest |J - y| at y0, given a positive multiplier, so that the perturbation
    reaches the state (by 7e-5 .. 2e-4 of max|y| in the float64 oracle, 7x .. 17x the bound)."""
    _check_tier(c)
    _, _, ncta, gpc = resident_plan(_lib(), _num_sms(), c.G, c.H, c.n, c.adjoint)
    w, y0, t, target = _inputs(c, 5500 + c.H)
    lo = (ncta - 1) * gpc
    n_loc = c.G - lo
    drift = (O.rhs(w, y0, decay=False) - y0).reshape(-1).abs()
    g = max(range(lo + min(15, n_loc - 1), c.G, 16), key=lambda r: float(drift[r]))
    w.gene_multipliers[0, g] = abs(float(w.gene_multipliers[0, g])) + 0.5
    bad_w = O.Weights(*[p.clone() for p in w.as_list()])
    bad_w.Wa[g] *= 1 + 1e-3
    y, _, _, _, _ = _run(pb, c, make_net(pb, bad_w), y0, t, target)
    y_ref, _, _, _ = _reference(w, y0, t, target, c.method, False, c.kernel)
    assert rel_l2(y, y_ref) < L2_TOL, "relative L2 alone should not see one row at this size"
    assert mismatches("y", y, y_ref, C_STATE), "one wrong WA row went unnoticed"
    assert int((y.double() - y_ref).abs().reshape(-1, c.G).amax(0).argmax()) == g
    # and the same call with the right weights passes (the rejection is the row's doing)
    y_ok, _, _, _, _ = _run(pb, c, make_net(pb, w), y0, t, target)
    assert not mismatches("y", y_ok, y_ref, C_STATE)
