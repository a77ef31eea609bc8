"""Forward + backward through odeint_adjoint_many with the fixed-grid step size (options=dict(step_size=h), rk4) against
dopri5 at rtol 1e-7 / atol 1e-9, one output interval of length dt per sample (the training step):

    yeast-5     yeast 3 551 x 120, 4 samples, dt 5
    yeast-10    yeast 3 551 x 120, 4 samples, dt 10
    breast      breast 11 165 x 200, 17 samples, dt 1 (the bench.py weights)

    python tools/step_size_timing.py [--reps 10] [--out FILE]

rk4 runs with step_size = dt (one step per interval, the same grid as no step size), dt / 4 and dt / 16.  The sample
start times are multiples of 1/8, so that every grid point is exact and the grid ends on t1 (a random start can leave
the last point of a float64 grid one ulp short of t1, which the reference refuses with an AssertionError).  A timed
repetition is one forward + one backward (CUDA events around both, all variants alternating within every repetition).
The error column is the relative L2 distance of y(t1) from a float64 dopri5 solve of the oracle (rtol 1e-10), over the
first four samples (the float64 solves run on the CPU).  RHS evaluations per sample are the forward's status n_rhs.
Prints the card's name and power limit with the medians.  Needs a GPU."""
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
from oracle import phoenix_oracle as O  # noqa: E402

# (name, G, H, samples, dt)
WORKLOADS = [("yeast-5", 3551, 120, 4, 5.0), ("yeast-10", 3551, 120, 4, 10.0), ("breast", bench.G, bench.H, bench.BATCH, 1.0)]


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as exc:   # the timing stands without it, but say so
        return "nvidia-smi unavailable (%s)" % exc


def variants(dt):
    return [("dopri5", "dopri5", None), ("rk4 h=dt", "rk4", dt), ("rk4 h=dt/4", "rk4", dt / 4),
            ("rk4 h=dt/16", "rk4", dt / 16)]


def workload(name, G, H, N, DT, reps, out):
    torch.manual_seed(0)
    net = pb.ODENet("cuda", G, neurons=H)
    if G == bench.G and H == bench.H:
        with torch.no_grad():
            for p, src in zip(net.parameters(), bench.synthetic_weights(0, dense=False)):
                p.copy_(src.reshape(p.shape))
    gen = torch.Generator().manual_seed(1)
    y0 = torch.rand(N, 1, G, generator=gen).cuda()
    t = (torch.arange(N, dtype=torch.float64) % 8 / 8).unsqueeze(1) + torch.tensor([0.0, DT], dtype=torch.float64)
    target = torch.rand(N, 1, G, generator=gen).cuda()
    vs = variants(DT)

    def once(method, h):
        net.zero_grad(set_to_none=True)
        opts = None if h is None else dict(step_size=h)
        y = pb.odeint_adjoint_many(net, y0, t, method=method, options=opts)
        torch.mean((y[:, 1] - target) ** 2).backward()
        return y.detach()

    # float64 reference of y(t1) and each variant's distance from it
    wd = O.Weights(*[p.detach().double().cpu() for p in net.parameters()])   # (reference parameter order and shapes)
    NE = min(N, 4)
    ref = torch.stack([O.odeint(wd, y0[i].double().cpu(), t[i], method="dopri5", rtol=1e-10, atol=1e-12)[0][1]
                       for i in range(NE)])
    info = {}
    for label, method, h in vs:
        y = once(method, h)
        with torch.no_grad():
            pb.engine.solve_forward(net, y0[0], t[0].tolist(), False, False, method, 1e-7, 1e-9, 2 ** 31 - 1,
                                    **({} if h is None else {"step_size": h}))
        n_rhs = pb.engine.last_status()["n_rhs"]
        err = float((y[:NE, 1].double().cpu() - ref).norm() / ref.norm())
        info[label] = (n_rhs, err)
    for _ in range(2):   # warm-up
        for _, method, h in vs:
            once(method, h)
    times = {label: [] for label, _, _ in vs}
    for _ in range(reps):
        for label, method, h in vs:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            once(method, h)
            b.record()
            torch.cuda.synchronize()
            times[label].append(a.elapsed_time(b))
    for label, _, _ in vs:
        n_rhs, err = info[label]
        line = "%-9s G=%-5d H=%-3d N=%-2d dt=%-4g %-12s fwd RHS/sample %4d  fwd+bwd %8.3f ms (median of %d)  " \
               "y(t1) rel-L2 vs float64 %.2e" % (name, G, H, N, DT, label, n_rhs, statistics.median(times[label]), reps, err)
        print(line)
        out.append(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("step_size_timing needs a GPU")
    lines = ["card: " + card()]
    print(lines[0])
    for w in WORKLOADS:
        workload(*w, a.reps, lines)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
