"""CPU: pin oracle/phoenix_oracle.py against the golden vectors generated from the reference itself."""
import pytest
import torch

from oracle import phoenix_oracle as O
from golden_util import (assert_logs_close, big_case_inputs, check_big_case, compare_logs, load, manifest,
                         manifest_big, rel_l2, weights_of)

RHS = [m["name"] for m in manifest("rhs")]
SOLVE = [m for m in manifest("solve")]


@pytest.fixture
def golden_threads():
    """Sets the number of torch CPU threads for one test.  MKL splits the reductions of a matmul by thread count, so the
    bit-exact comparisons run with the counts the goldens were generated with (tests/golden/make_golden.py): 8 for the
    RHS cases, 1 for the stored solves."""
    saved = torch.get_num_threads()
    yield torch.set_num_threads
    torch.set_num_threads(saved)


@pytest.mark.parametrize("name", RHS)
def test_rhs_and_vjp_match_reference_autograd(name, golden_threads):
    golden_threads(8)
    d = load(name)
    w = weights_of(d)
    y, g = torch.from_numpy(d["y"]), torch.from_numpy(d["g"])
    for tag, decay in (("decay", True), ("prior", False)):
        f = O.rhs(w, y, decay=decay)
        # same ATen kernels as the reference -> bit-exact forward
        assert torch.equal(f, torch.from_numpy(d["f_" + tag])), (name, tag)
        f2, ybar, pbar = O.rhs_vjp(w, y, g, decay=decay)
        assert torch.equal(f2, f)
        assert rel_l2(ybar, d["ybar_" + tag]) < 2e-6
        for i, p in enumerate(pbar):
            ref = d["pbar%d_%s" % (i, tag)]
            assert rel_l2(p, ref) < 2e-6, (name, tag, i)


@pytest.mark.parametrize("m", SOLVE, ids=[m["name"] for m in SOLVE])
def test_solve_and_adjoint_match_reference(m, golden_threads):
    golden_threads(1)
    d = load(m["name"])
    w = weights_of(d)
    y0, t = torch.from_numpy(d["y0"]), torch.from_numpy(d["t"])
    rtol, atol = float(d["rtol"]), float(d["atol"])
    loose = rtol > 1e-6
    y, flog = O.odeint(w, y0, t, method=m["method"], rtol=rtol, atol=atol)
    if m["method"] == "dopri5":
        n, msg = compare_logs(flog.steps, d["flog"], dt_rtol=2e-2 if loose else 1e-6)
        if int(d["stable"]) and not loose:
            assert msg == "identical", msg   # same ATen kernels as the reference -> identical forward sequence
        assert_logs_close(flog.steps, d["flog"], 5e-2, m["name"])
        assert rel_l2(y, d["y"]) < (1e-5 if loose else 1e-6)
    else:
        assert torch.equal(y, torch.from_numpy(d["y"]))
    if not m["adjoint"]:
        return
    target = torch.from_numpy(d["target"])
    loss = torch.mean((y[1:] - target) ** 2)
    assert abs(loss.item() - float(d["loss"])) <= 1e-6 * abs(float(d["loss"]))
    grad_y = torch.zeros_like(y)
    grad_y[1:] = 2.0 * (y[1:] - target) / target.numel()
    ady, grads, blog = O.adjoint_backward(w, t, y, grad_y, method=m["method"], rtol=rtol, atol=atol)
    tol = 1e-5 if m["method"] != "dopri5" else (5e-3 if loose else 3e-5)
    assert rel_l2(ady, d["adj_y0"]) < tol
    for i, g in enumerate(grads):
        assert rel_l2(g, d["grad%d" % i]) < tol, (m["name"], i, rel_l2(g, d["grad%d" % i]))
    if m["method"] == "dopri5" and loose:
        assert_logs_close(blog.steps, d["blog"], 5e-2, m["name"])
    elif m["method"] == "dopri5" and int(d["stable"]):
        n, msg = compare_logs(blog.steps, d["blog"], dt_rtol=1e-4)
        # the explicit-formula VJP differs from autograd by rounding only; a mismatch here is reported, and is an
        # error only if the values above also failed
        print(m["name"], "adjoint step log vs reference:", msg)


BIG = manifest_big()


@pytest.mark.parametrize("m", BIG, ids=[m["name"] for m in BIG])
def test_baseline_configs_on_real_data_match_reference(m):
    """C3 (yeast, real 24-point series, dt = 5 / 10) and C4 (breast, real rows, dt = 0.0051): the per-sample loop of
    training_step (train_insilico.py:128-138) restated with the oracle against the reference's own outputs."""
    d = load(m["name"])
    w, y0, t, target = big_case_inputs(m, d)
    preds, flogs = [], []
    for i in range(m["N"]):
        y, fl = O.odeint(w, y0[i], t[i], method=m["method"])
        preds.append(y)
        flogs.append(fl.steps)
    pred = torch.stack([y[1] for y in preds])
    loss, gpred = O.mse_loss_and_grad(pred, target)
    adys, total = [], None
    for i in range(m["N"]):
        gy = torch.zeros_like(preds[i])
        gy[1] = gpred[i]
        ady, grads, bl = O.adjoint_backward(w, t[i], preds[i], gy, method=m["method"])
        adys.append(ady)
        total = grads if total is None else [a + b for a, b in zip(total, grads)]
        if m["method"] == "dopri5" and m["stable"]:
            assert compare_logs(flogs[i], d["flog%d" % i], 1e-6)[1] == "identical"
            assert compare_logs(bl.steps, d["blog%d" % i], 1e-4)[1] == "identical"
    dop = m["method"] == "dopri5"
    check_big_case(m, d, pred, loss, torch.stack(adys), total, 1e-6 if m["stable"] else 1e-5,
                   (3e-5 if m["stable"] else 2e-4) if dop else 1e-5)


def test_single_output_time_is_the_initial_state():
    """len(t) == 1 (solvers.py:26-30, adjoint.py:137-162: both loops are empty): y0 is the only slice, its cotangent is
    grad_y[0], the parameter cotangents are zero.  Checked against the reference itself for dopri5 / rk4 / euler when this
    case was added; the CUDA path is held to the same answers in tests/test_gpu_parity.py."""
    w = O.make_weights(20, 4, 1, dense=True)
    y0 = torch.rand(2, 1, 20, generator=torch.Generator().manual_seed(0))
    for method in ("dopri5", "rk4", "euler", "midpoint"):
        for dt in (torch.float32, torch.float64):
            t = torch.tensor([0.3], dtype=dt)
            y, _ = O.odeint(w, y0, t, method=method)
            assert y.shape == (1, 2, 1, 20) and torch.equal(y[0], y0)
            gy = torch.rand(1, 2, 1, 20, generator=torch.Generator().manual_seed(1))
            ady, grads, _ = O.adjoint_backward(w, t, y, gy, method=method)
            assert torch.equal(ady, gy[0])
            assert len(grads) == 6 and all(not g.any() for g in grads)
