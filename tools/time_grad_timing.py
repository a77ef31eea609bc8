"""Forward + backward through odeint_adjoint_many (the training step's sweeps), dopri5 at rtol 1e-7 / atol 1e-9, one output
interval per sample, with t not requiring grad against t requiring grad (t.grad from phx_time_vjp, and the time
cotangents in the backward's initial step):

    bench       breast 11 165 x 200, 17 samples, dt 0.0051 (the bench.py workload and inputs)
    yeast       yeast 3 551 x 120, 17 samples, dt 5

    python tools/time_grad_timing.py [--reps 20] [--out FILE]

CUDA events around forward + loss + backward; the two variants alternate within every repetition so that they share the
same clocks.  Backward attempts / rejections per variant come from the step logs of a separate logged call; rel-L2 of
adj_y0 and of the parameter gradients against the run without t grad (the time cotangent can move the first backward
dt).  Prints the card's name and power limit with the medians.  Needs a GPU."""
import argparse
import os
import statistics
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import torch  # noqa: E402

import bench  # noqa: E402
import phoenix_b200 as pb  # noqa: E402

# (name, G, H, samples, dt)
WORKLOADS = [("bench", bench.G, bench.H, bench.BATCH, bench.DT), ("yeast", 3551, 120, 17, 5.0)]


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as exc:   # the timing stands without it, but say so
        return "nvidia-smi unavailable (%s)" % exc


def rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def workload(name, G, H, N, DT, reps):
    torch.manual_seed(0)
    net = pb.ODENet("cuda", G, neurons=H)
    if G == bench.G and H == bench.H:
        with torch.no_grad():
            for p, src in zip(net.parameters(), bench.synthetic_weights(0, dense=False)):
                p.copy_(src.reshape(p.shape))
    params = list(net.parameters())
    gen = torch.Generator().manual_seed(1)
    y0 = torch.rand(N, 1, G, generator=gen).cuda()
    t0 = torch.rand(N, 1, generator=gen, dtype=torch.float64)
    t_base = t0 + torch.tensor([0.0, DT], dtype=torch.float64)
    target = torch.rand(N, 1, G, generator=gen).cuda()

    def step(t_grad, logged=False):
        net.zero_grad(set_to_none=True)
        t = t_base.clone().requires_grad_(t_grad)
        y0g = y0.clone().requires_grad_(True)
        pb.set_step_logging(logged)
        try:
            y = pb.odeint_adjoint_many(net, y0g, t, method="dopri5")
            torch.mean((y[:, 1] - target) ** 2).backward()
            blog = [pb.last_step_log(i) for i in range(N)] if logged else None
        finally:
            pb.set_step_logging(False)
        return y0g.grad, [p.grad.clone() for p in params], t.grad, blog

    a_ref, g_ref, _, _ = step(False, True)
    variants = [("no-t-grad", False), ("t-grad", True)]
    lines = ["%s: %d x %d, %d samples, dt %g" % (name, G, H, N, DT)]
    stats = {}
    for nm, tg in variants:
        a, g, tgrad, bl = step(tg, True)
        ba, br = sum(len(x) for x in bl), sum(1 for x in bl for s in x if not s[2])
        stats[nm] = ("bwd attempts %d rejected %d; rel-L2 adj_y0 %.2e, grads max %.2e%s"
                     % (ba, br, rel(a, a_ref), max(rel(x, z) for x, z in zip(g, g_ref)),
                        "; |t.grad| %.3e" % float(tgrad.norm()) if tgrad is not None else ""))

    def once(tg):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step(tg)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    for _, tg in variants:   # warm-up: module load, workspaces
        once(tg)
        once(tg)
    times = {nm: [] for nm, _ in variants}
    for _ in range(reps):
        for nm, tg in variants:
            times[nm].append(once(tg))
    base = statistics.median(times["no-t-grad"])
    for nm, _ in variants:
        m = statistics.median(times[nm])
        lines.append("  %-9s median %.3f ms  min %.3f  max %.3f  (%.1f %% of no-t-grad)  %s"
                     % (nm, m, min(times[nm]), max(times[nm]), 100.0 * m / base, stats[nm]))
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_grad_timing: needs a GPU")
    pb.set_sync_errors(True)
    lines = ["Forward + backward through odeint_adjoint_many, t without / with requires_grad: CUDA events, %d alternated "
             "repetitions, dopri5 rtol 1e-7 / atol 1e-9" % args.reps, "card: %s" % card()]
    for w in WORKLOADS:
        lines += workload(*w, args.reps)
        print("\n".join(lines[-3:]), flush=True)
    text = "\n".join(lines)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
