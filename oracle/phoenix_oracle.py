"""CPU oracle for the PHOENIX NeuralODE hot path.  TEST INFRASTRUCTURE ONLY.

This file is a checker, not a product path: only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import it.  Nothing under ``phoenix_b200/``
imports it, and the product raises if its CUDA library is missing rather than falling back here.

It restates, on torch-CPU tensors (the reference's own arithmetic back-end: the same ATen fp32 kernels), the
algorithm of the reference's hot path:

* RHS  ``ODENet.forward`` / ``prior_only_forward``            -> ``rhs``            (odenet.py:21-35, 85-98)
* VJP  of the RHS (explicit formulas, no autograd)             -> ``rhs_vjp``        (adjoint.py:94-127 via autograd)
* fixed-grid ``euler`` / ``midpoint`` / ``rk4`` (3/8 rule)       -> ``_solve_fixed``   (solvers.py:77-103, fixed_grid.py:6-38,
                                                                                    rk_common.py:96-103)
* adaptive ``dopri5``                                          -> ``_solve_dopri5``  (rk_common.py:39-77,111-228, dopri5.py:5-36,
                                                                                    interp.py:1-47, misc.py:47-103)
* the adjoint backward sweep on the flattened augmented state  -> ``adjoint_backward`` (adjoint.py:32-162, misc.py:14-44,145-162)

Parity pinning: the reference has no tests or golden vectors of its own (SURVEY.md section 4), so this oracle is
pinned against outputs of the reference itself, generated in the build container by
``tests/golden/make_golden.py`` (which imports ``/root/reference/ode_net/code``) and committed as
``tests/golden/*.npz``.  ``tests/test_oracle_golden.py`` checks every function here against those vectors.

Parameter order everywhere is the reference's ``ODENet.parameters()`` order (SURVEY.md appendix A):
``gene_multipliers [1,G]``, ``Wp [H,G]``, ``bp [H]``, ``Ws [H,G]``, ``bs [H]``, ``Wa [G,2H]``.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Callable, List, Optional, Sequence, Tuple

import torch

PARAM_ORDER = ("gene_multipliers", "Wp", "bp", "Ws", "bs", "Wa")


@dataclass
class Weights:
    """The six trainable tensors of the PHOENIX RHS, fp32, reference shapes (odenet.py:49-61)."""

    gene_multipliers: torch.Tensor  # [1, G]
    Wp: torch.Tensor  # [H, G]   net_prods.linear_out.weight
    bp: torch.Tensor  # [H]      net_prods.linear_out.bias
    Ws: torch.Tensor  # [H, G]   net_sums.linear_out.weight
    bs: torch.Tensor  # [H]      net_sums.linear_out.bias
    Wa: torch.Tensor  # [G, 2H]  net_alpha_combine.linear_out.weight (no bias)

    def as_list(self) -> List[torch.Tensor]:
        return [getattr(self, n) for n in PARAM_ORDER]

    @property
    def G(self) -> int:
        return self.Ws.shape[1]

    @property
    def H(self) -> int:
        return self.Ws.shape[0]

    @property
    def P(self) -> int:
        return sum(p.numel() for p in self.as_list())


def make_weights(G: int, H: int, seed: int, dense: bool = False, neg_mult_frac: float = 0.0) -> Weights:
    """Synthetic weights with the reference's init distribution (odenet.py:61-75, SURVEY.md a5).

    ``dense=False``: ``nn.init.sparse_(sparsity=0.95, std=0.05)`` (per column 95 % zeros) for the three matrices,
    ``nn.Linear`` default biases U(+-1/sqrt(fan_in)), multipliers U[0,1).  ``dense=True``: matrices N(0, 0.05^2)
    ("trained-like").  ``neg_mult_frac`` flips that fraction of multipliers negative to exercise the relu mask.
    """
    gen = torch.Generator().manual_seed(seed)

    def mat(rows: int, cols: int) -> torch.Tensor:
        w = torch.randn(rows, cols, generator=gen) * 0.05
        if not dense:
            nz = int(math.ceil(0.95 * rows))
            for c in range(cols):
                idx = torch.randperm(rows, generator=gen)[:nz]
                w[idx, c] = 0.0
        return w.contiguous()

    Ws = mat(H, G)
    Wp = mat(H, G)
    Wa = mat(G, 2 * H)
    bound = 1.0 / math.sqrt(G)
    bs = (torch.rand(H, generator=gen) * 2 - 1) * bound
    bp = (torch.rand(H, generator=gen) * 2 - 1) * bound
    m = torch.rand(1, G, generator=gen)
    if neg_mult_frac > 0:
        flip = torch.rand(1, G, generator=gen) < neg_mult_frac
        m = torch.where(flip, -m, m)
    return Weights(m.float(), Wp.float(), bp.float(), Ws.float(), bs.float(), Wa.float())


# --------------------------------------------------------------------------------------------------------------
# RHS and its VJP
# --------------------------------------------------------------------------------------------------------------

def hill_terms(y: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """(s, l, den): soft-sign of the shifted input, its log1p, and 1+|y-0.5| (odenet.py:21-25, 31-35)."""
    z = y - 0.5
    den = 1 + torch.abs(z)
    s = z / den
    return s, torch.log1p(s), den


def rhs(w: Weights, y: torch.Tensor, decay: bool = True) -> torch.Tensor:
    """f(y) of odenet.py:85-91 (``decay=True``) or the pre-decay ``joint`` of odenet.py:93-98 (``decay=False``)."""
    s, l, _ = hill_terms(y)
    S = torch.nn.functional.linear(s, w.Ws, w.bs)
    Pr = torch.exp(torch.nn.functional.linear(l, w.Wp, w.bp))
    J = torch.nn.functional.linear(torch.cat((S, Pr), dim=-1), w.Wa)
    if not decay:
        return J
    return torch.relu(w.gene_multipliers) * (J - y)


def rhs_vjp(w: Weights, y: torch.Tensor, g: torch.Tensor, decay: bool = True):
    """(f, ybar, [6 parameter cotangents]) for cotangent ``g`` of f — SURVEY.md a15 formulas (checked there in fp64
    against autograd).  Shapes: y, g ``[..., G]``; leading dims are flattened into B rows."""
    G, H = w.G, w.H
    y2 = y.reshape(-1, G)
    g2 = g.reshape(-1, G)
    s, l, den = hill_terms(y2)
    S = torch.nn.functional.linear(s, w.Ws, w.bs)
    Pr = torch.exp(torch.nn.functional.linear(l, w.Wp, w.bp))
    SP = torch.cat((S, Pr), dim=-1)
    J = torch.nn.functional.linear(SP, w.Wa)
    if decay:
        rm = torch.relu(w.gene_multipliers)
        f = rm * (J - y2)
        gJ = g2 * rm
        mbar = (g2 * (J - y2)).sum(0, keepdim=True) * (w.gene_multipliers > 0).to(y2.dtype)
    else:
        f = J
        gJ = g2
        mbar = torch.zeros_like(w.gene_multipliers)
    Wabar = gJ.t() @ SP
    gSP = gJ @ w.Wa
    gS = gSP[:, :H]
    gLP = gSP[:, H:] * Pr
    bsbar = gS.sum(0)
    bpbar = gLP.sum(0)
    Wsbar = gS.t() @ s
    Wpbar = gLP.t() @ l
    ybar = (gS @ w.Ws + (gLP @ w.Wp) / (1 + s)) / (den * den)
    if decay:
        ybar = ybar - gJ
    return f.reshape(y.shape), ybar.reshape(y.shape), [mbar, Wpbar, bpbar, Wsbar, bsbar, Wabar]


# --------------------------------------------------------------------------------------------------------------
# Dormand-Prince 5(4) tableau (dopri5.py:5-30), kept in float64 and cast to the state dtype at use
# --------------------------------------------------------------------------------------------------------------
DP_ALPHA = [1 / 5, 3 / 10, 4 / 5, 8 / 9, 1.0, 1.0]
DP_BETA = [
    [1 / 5],
    [3 / 40, 9 / 40],
    [44 / 45, -56 / 15, 32 / 9],
    [19372 / 6561, -25360 / 2187, 64448 / 6561, -212 / 729],
    [9017 / 3168, -355 / 33, 46732 / 5247, 49 / 176, -5103 / 18656],
    [35 / 384, 0, 500 / 1113, 125 / 192, -2187 / 6784, 11 / 84],
]
DP_C_ERROR = [
    35 / 384 - 1951 / 21600,
    0,
    500 / 1113 - 22642 / 50085,
    125 / 192 - 451 / 720,
    -2187 / 6784 - -12231 / 42400,
    11 / 84 - 649 / 6300,
    -1.0 / 60.0,
]
DP_C_MID = [
    6025192743 / 30085553152 / 2,
    0,
    51252292925 / 65400821598 / 2,
    -2691868925 / 45128329728 / 2,
    187940372067 / 1594534317056 / 2,
    -1776094331 / 19743644256 / 2,
    11237099 / 235043384 / 2,
]


def rms(x: torch.Tensor) -> torch.Tensor:
    """misc.py:10-11."""
    return x.pow(2).mean().sqrt()


def block_max_rms(sizes: Sequence[int]) -> Callable[[torch.Tensor], torch.Tensor]:
    """max over consecutive blocks of the RMS of each block (misc.py:14-24 / 27-40 with rms per block)."""

    def norm(x: torch.Tensor) -> torch.Tensor:
        out, lo = [], 0
        for n in sizes:
            out.append(rms(x[lo:lo + n]))
            lo += n
        assert lo == x.numel()
        return max(out)

    return norm


@dataclass
class StepLog:
    """(t0, dt, accepted) per attempted adaptive step, plus RHS-evaluation count.  dopri5 also records the error ratio
    it computes for each attempt and, per solve, (index of its first attempt, Hairer's initial step estimate)."""

    steps: List[Tuple[float, float, bool]]
    nfe: int = 0
    ratios: List[float] = field(default_factory=list)
    starts: List[Tuple[int, float]] = field(default_factory=list)


class Replay:
    """A step schedule ``(t0, dt, accepted)`` per attempt -- the rows of ``engine.last_step_log()`` -- that dopri5 solves
    consume in order in place of their step-size controller (``_solve_dopri5``).  ``finish()`` checks that every attempt
    was used."""

    def __init__(self, steps):
        self.steps = [(float(a), float(b), bool(c)) for a, b, c in steps]
        self.pos = 0

    def take(self, t1: float) -> Tuple[float, bool]:
        assert self.pos < len(self.steps), "replay: the schedule ends at attempt %d, before the solve does" % self.pos
        t0, dt, acc = self.steps[self.pos]
        assert abs(t0 - t1) <= 1e-12 * (abs(t1) + abs(dt)), \
            "replay: attempt %d starts at %r, the last accepted step ended at %r" % (self.pos, t0, t1)
        assert dt != 0 and math.isfinite(dt), "replay: attempt %d has dt %r" % (self.pos, dt)
        self.pos += 1
        return dt, acc

    def finish(self):
        assert self.pos == len(self.steps), "replay: %d of %d attempts left over" % (len(self.steps) - self.pos,
                                                                                 len(self.steps))


def _initial_step(func, t0, y0, f0, rtol, atol, norm) -> torch.Tensor:
    """Hairer's starting step with order-1 = 4 (misc.py:47-86).  rtol/atol are 0-dim float64 tensors; every
    intermediate stays in the state dtype exactly as in the reference."""
    dtype = y0.dtype
    t_dtype = t0.dtype
    t0s = t0.to(dtype)
    scale = atol + torch.abs(y0) * rtol
    d0 = norm(y0 / scale)
    d1 = norm(f0 / scale)
    if d0 < 1e-5 or d1 < 1e-5:
        h0 = torch.tensor(1e-6, dtype=dtype)
    else:
        h0 = 0.01 * d0 / d1
    f1 = func(t0s + h0, y0 + h0 * f0)
    d2 = norm((f1 - f0) / scale) / h0
    if d1 <= 1e-15 and d2 <= 1e-15:
        h1 = torch.max(torch.tensor(1e-6, dtype=dtype), h0 * 1e-3)
    else:
        h1 = (0.01 / max(d1, d2)) ** (1.0 / 5.0)
    return torch.min(100 * h0, h1).to(t_dtype)


def _next_dt(dt: torch.Tensor, ratio: torch.Tensor) -> torch.Tensor:
    """misc.py:94-103 with safety 0.9, ifactor 10, dfactor 0.2, order 5 (rk_common.py:116)."""
    if ratio == 0:
        return dt * 10.0
    dfactor = 1.0 if ratio < 1 else 0.2
    r = ratio.to(dt.dtype)
    factor = min(10.0, max(0.9 / float(r ** torch.tensor(0.2, dtype=dt.dtype)), dfactor))
    if math.isnan(float(r)):
        factor = float("nan")
    return dt * factor


def _solve_dopri5(func, y0: torch.Tensor, t: torch.Tensor, rtol: float, atol: float, norm, log: StepLog,
                  max_num_steps: int = 2 ** 31 - 1, replay: Optional[Replay] = None) -> torch.Tensor:
    """Adaptive Dormand-Prince solve returning y at every t (rk_common.py:140-228, solvers.py:23-30).

    State dtype = y0.dtype (fp32); every time-like scalar is a 0-dim float64 tensor; the stage matrix ``k`` has the
    stage index innermost and stage combinations are ``k[..., :i+1] @ (beta_i * dt)`` as in rk_common.py:62-76.

    ``replay``: take each attempt's dt and accept decision from the schedule instead of Hairer's estimate, the
    controller and ``ratio <= 1``; everything else runs as without it (the estimate and the ratios are still computed
    and logged).  The schedule must be one a solve of these output times can take: each attempt starts where the last
    accepted step ended, so the first one at t[0], and no attempt follows the step that covers the last output time."""
    dtype = y0.dtype
    t = t.to(torch.float64)
    rt = torch.as_tensor(rtol, dtype=torch.float64)
    at = torch.as_tensor(atol, dtype=torch.float64)
    beta = [torch.tensor(b, dtype=torch.float64).to(dtype) for b in DP_BETA]
    c_err = torch.tensor(DP_C_ERROR, dtype=torch.float64).to(dtype)
    c_mid = torch.tensor(DP_C_MID, dtype=torch.float64).to(dtype)

    def f(tt, yy):
        log.nfe += 1
        return func(tt.to(dtype), yy)

    out = torch.empty(len(t), *y0.shape, dtype=dtype)
    out[0] = y0
    f0 = f(t[0], y0)
    dt = _initial_step(f, t[0], y0, f0, rt, at, norm)
    log.starts.append((len(log.steps), float(dt)))
    y, t0, t1 = y0, t[0], t[0]
    coeff = [y0] * 5
    for i in range(1, len(t)):
        n = 0
        while t[i] > t1:
            assert n < max_num_steps, "max_num_steps exceeded ({}>={})".format(n, max_num_steps)
            if replay is not None:
                dt_r, accept_r = replay.take(float(t1))
                dt = torch.tensor(dt_r, dtype=torch.float64)
            assert t1 + dt > t1, "underflow in dt {}".format(dt.item())
            assert torch.isfinite(y).all(), "non-finite values in state `y`: {}".format(y)
            ts, dts = t1.to(dtype), dt.to(dtype)
            k = torch.empty(*f0.shape, 7, dtype=dtype)
            k[..., 0] = f0
            for s_idx in range(6):
                yi = y + k[..., :s_idx + 1].matmul(beta[s_idx] * dts).view_as(f0)
                k[..., s_idx + 1] = f(ts + DP_ALPHA[s_idx] * dts, yi)
            y1, f1 = yi, k[..., 6]
            err = k.matmul(dts * c_err)
            tol = at + rt * torch.max(y.abs(), y1.abs())
            ratio = norm(err / tol)
            accept = bool(ratio <= 1) if replay is None else accept_r
            log.steps.append((float(t1), float(dt), accept))
            log.ratios.append(float(ratio))
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
            dt = _next_dt(dt, ratio)
            n += 1
        # quartic dense output on the last accepted step (interp.py:25-47)
        assert (t0 <= t[i]) & (t[i] <= t1), "invalid interpolation"
        x = (t[i] - t0) / (t1 - t0)
        total = coeff[0] + x * coeff[1]
        xp = x
        for c in coeff[2:]:
            xp = xp * x
            total = total + xp * c
        out[i] = total
    return out


def _solve_fixed(func, y0: torch.Tensor, t: torch.Tensor, method: str, log: StepLog) -> torch.Tensor:
    """One step per output interval, grid == t (solvers.py:48-50, 77-95); euler fixed_grid.py:13-14, midpoint
    :24-27, rk4 = 3/8 rule rk_common.py:96-103."""
    out = torch.empty(len(t), *y0.shape, dtype=y0.dtype)
    out[0] = y0
    y = y0

    def f(tt, yy):
        log.nfe += 1
        return func(tt, yy)

    for i in range(len(t) - 1):
        t0, dt = t[i], t[i + 1] - t[i]
        if method == "euler":
            dy = dt * f(t0, y)
        elif method == "midpoint":
            half = 0.5 * dt
            dy = dt * f(t0 + half, y + f(t0, y) * half)
        elif method == "rk4":
            k1 = f(t0, y)
            k2 = f(t0 + dt / 3, y + dt * k1 * (1 / 3))
            k3 = f(t0 + dt * (2 / 3), y + dt * (k2 - k1 * (1 / 3)))
            k4 = f(t0 + dt, y + dt * (k1 - k2 + k3))
            dy = (k1 + 3 * (k2 + k3) + k4) * dt * 0.125
        else:
            raise ValueError('Invalid method "{}"'.format(method))
        y = y + dy
        out[i + 1] = y
    return out


def _solve(func, y0, t, method, rtol, atol, norm, log, replay=None):
    if method is None:
        method = "dopri5"
    assert t.ndim == 1 and bool((t[1:] > t[:-1]).all()), "t must be strictly increasing here"
    if method == "dopri5":
        return _solve_dopri5(func, y0, t, rtol, atol, norm, log, replay=replay)
    assert replay is None, "a step schedule is for dopri5"
    return _solve_fixed(func, y0, t, method, log)


def odeint(w: Weights, y0: torch.Tensor, t: torch.Tensor, method: Optional[str] = None, rtol: float = 1e-7,
           atol: float = 1e-9, replay=None) -> Tuple[torch.Tensor, StepLog]:
    """Forward solve ``[len(t), *y0.shape]`` with the reference defaults (odeint.py:25; norm = RMS over the whole
    state, misc.py:198-201).  Decreasing ``t`` is handled by time negation as misc.py:210-218.  ``replay``: a dopri5
    step log to take instead of the controller's steps (``Replay``)."""
    log = StepLog([])
    sign = 1.0
    if bool((t[1:] < t[:-1]).all()):
        sign, t = -1.0, -t
    func = (lambda tt, yy: rhs(w, yy)) if sign > 0 else (lambda tt, yy: -rhs(w, yy))
    rp = None if replay is None else Replay(replay)
    with torch.no_grad():
        y = _solve(func, y0, t, method, rtol, atol, rms, log, rp)
    if rp is not None:
        rp.finish()
    return y, log


def adjoint_backward(w: Weights, t: torch.Tensor, y: torch.Tensor, grad_y: torch.Tensor,
                     method: Optional[str] = None, rtol: float = 1e-7, atol: float = 1e-9, replay=None):
    """The backward sweep of ``OdeintAdjointMethod`` (adjoint.py:32-162) for increasing ``t``.

    For each output interval, from the last to the first, the flat augmented vector
    ``[vjp_t(1), y(N), adj_y(N), adj_params(P)]`` is integrated from t[i] to t[i-1] in negated time
    (misc.py:210-212) with the forward method and tolerances, under the norm
    ``max(RMS(vjp_t), RMS(y), RMS(adj_y), RMS(adj_params))`` (adjoint.py:72-78 / 198-200).  ``vjp_t`` stays 0
    because t does not require grad.  ``replay``: a dopri5 backward step log, the attempts of all intervals in the
    order they run (T-1 .. 1, negated time), taken instead of the controller's steps (``Replay``).  Returns (adj_y0,
    [6 grads], StepLog over all intervals)."""
    log = StepLog([])
    shape = y.shape[1:]
    N = y[0].numel()
    params = w.as_list()
    psz = [p.numel() for p in params]
    P = sum(psz)
    norm = block_max_rms([1, N, N, P])

    def aug_reversed(tt, z):
        yy = z[1:1 + N].reshape(shape)
        aa = z[1 + N:1 + 2 * N].reshape(shape)
        f, ybar, pbar = rhs_vjp(w, yy, -aa)
        full = torch.cat([torch.zeros(1, dtype=z.dtype), f.reshape(-1), ybar.reshape(-1)]
                         + [p.reshape(-1) for p in pbar])
        return -full

    rp = None if replay is None else Replay(replay)
    with torch.no_grad():
        adj_y = grad_y[-1].clone()
        adj_p = torch.zeros(P, dtype=y.dtype)
        cur_y = y[-1]
        for i in range(len(t) - 1, 0, -1):
            z0 = torch.cat([torch.zeros(1, dtype=y.dtype), cur_y.reshape(-1), adj_y.reshape(-1), adj_p])
            tt = -t[i - 1:i + 1].flip(0)
            z = _solve(aug_reversed, z0, tt, method, rtol, atol, norm, log, rp)[1]
            adj_p = z[1 + 2 * N:]
            cur_y = y[i - 1]
            adj_y = z[1 + N:1 + 2 * N].reshape(shape) + grad_y[i - 1]
        if rp is not None:
            rp.finish()
        grads, lo = [], 0
        for p, n in zip(params, psz):
            grads.append(adj_p[lo:lo + n].reshape(p.shape))
            lo += n
    return adj_y, grads, log


def mse_loss_and_grad(pred: torch.Tensor, target: torch.Tensor):
    """loss = mean((pred-target)^2) and d loss / d pred (train_insilico.py:132)."""
    diff = pred - target
    return (diff * diff).mean(), 2.0 * diff / diff.numel()
