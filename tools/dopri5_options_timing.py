"""Forward + backward through odeint_adjoint_many (the training step's sweeps), dopri5 at rtol 1e-7 / atol 1e-9, one output
interval per sample, without options against options=dict(first_step=h) (inherited by the backward):

    bench       breast 11 165 x 200, 17 samples, dt 0.0051 (the bench.py workload and inputs)
    breast-1    breast 11 165 x 200, 17 samples, dt 1.0
    yeast       yeast 3 551 x 120, 17 samples, dt 5

    python tools/dopri5_options_timing.py [--reps 20] [--out FILE]

h is the median over the samples of Hairer's estimate in the forward without options ("hairer"), and dt itself ("dt").
CUDA events around forward + loss + backward; the variants alternate within every repetition so that they share the
same clocks.  Attempts / rejections and RHS evaluations per sample (Hairer: 2 + 6 per attempt, first_step: 1 + 6 per
attempt) come from the step logs of a separate logged call; rel-L2 of y(t1) and of the gradients against the run without
options.  Prints the card's name and power limit with the medians.  Needs a GPU."""
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
WORKLOADS = [("bench", bench.G, bench.H, bench.BATCH, bench.DT), ("breast-1", bench.G, bench.H, bench.BATCH, 1.0),
             ("yeast", 3551, 120, 17, 5.0)]


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
    t = t0 + torch.tensor([0.0, DT], dtype=torch.float64)
    target = torch.rand(N, 1, G, generator=gen).cuda()

    def step(opts, logged=False):
        net.zero_grad(set_to_none=True)
        pb.set_step_logging(logged)
        try:
            y = pb.odeint_adjoint_many(net, y0, t, method="dopri5", options=opts)
            flog = [pb.last_step_log(i) for i in range(N)] if logged else None
            torch.mean((y[:, 1] - target) ** 2).backward()
            blog = [pb.last_step_log(i) for i in range(N)] if logged else None
        finally:
            pb.set_step_logging(False)
        return y.detach()[:, 1], [p.grad.clone() for p in params], flog, blog

    y_ref, g_ref, flog, _ = step(None, True)
    h = statistics.median(log[0][1] for log in flog)
    variants = [("none", None), ("hairer", dict(first_step=h)), ("dt", dict(first_step=DT))]
    lines = ["%s: %d x %d, %d samples, dt %g; median Hairer estimate of the forward %.6g" % (name, G, H, N, DT, h)]
    stats = {}
    for nm, opts in variants:
        y, g, fl, bl = step(opts, True)
        init = 2 if opts is None else 1
        fa, fr = sum(len(x) for x in fl), sum(1 for x in fl for s in x if not s[2])
        ba, br = sum(len(x) for x in bl), sum(1 for x in bl for s in x if not s[2])
        stats[nm] = ("fwd attempts %d rejected %d RHS/sample %.1f; bwd attempts %d rejected %d RHS/sample %.1f; "
                     "rel-L2 y(t1) %.2e, grads max %.2e"
                     % (fa, fr, init + 6 * fa / N, ba, br, init + 6 * ba / N, rel(y, y_ref),
                        max(rel(a, b) for a, b in zip(g, g_ref))))

    def once(opts):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step(opts)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    for _, opts in variants:   # warm-up: module load, workspaces
        once(opts)
        once(opts)
    times = {nm: [] for nm, _ in variants}
    for _ in range(reps):
        for nm, opts in variants:
            times[nm].append(once(opts))
    base = statistics.median(times["none"])
    for nm, _ in variants:
        m = statistics.median(times[nm])
        lines.append("  %-6s median %.3f ms  min %.3f  max %.3f  (%.1f %% of none)  %s"
                     % (nm, m, min(times[nm]), max(times[nm]), 100.0 * m / base, stats[nm]))
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dopri5_options_timing: needs a GPU")
    pb.set_sync_errors(True)
    lines = ["Forward + backward through odeint_adjoint_many, no options vs options=dict(first_step=h): CUDA events, %d "
             "alternated repetitions, dopri5 rtol 1e-7 / atol 1e-9" % args.reps, "card: %s" % card()]
    for w in WORKLOADS:
        lines += workload(*w, args.reps)
        print("\n".join(lines[-4:]), flush=True)
    text = "\n".join(lines)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
