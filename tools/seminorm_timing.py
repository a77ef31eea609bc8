"""Backward sweeps under the default error norm and under the seminorm (adjoint_options=dict(norm="seminorm")), all six
parameters in the adjoint set, dopri5 at rtol 1e-7 / atol 1e-9, one output interval per sample (the training step):

    bench       breast 11 165 x 200, 17 samples, dt 0.0051 (the bench.py workload and inputs)
    breast-1    breast 11 165 x 200, 17 samples, dt 1.0
    yeast       yeast 3 551 x 120, 4 samples, dt 5
    sim350      SIM350 350 x 40, 17 samples, dt 2

    python tools/seminorm_timing.py [--reps 20] [--out FILE]

One call of engine.solve_adjoint_many per timed sample, CUDA events around it; the two norms alternate within every
repetition so that they share the same clocks.  Backward attempted / rejected steps come from the step log of a separate
logged call; RHS evaluations per sample = 2 (Hairer's initial step) + 6 per attempt.  Prints the card's name and power
limit with the medians.  Needs a GPU."""
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
from phoenix_b200 import _lib, engine  # noqa: E402

NORMS = [("default", _lib.PARAMS_ALL), ("seminorm", _lib.PARAMS_ALL | _lib.NORM_SEMINORM)]
# (name, G, H, samples, dt)
WORKLOADS = [("bench", bench.G, bench.H, bench.BATCH, bench.DT), ("breast-1", bench.G, bench.H, bench.BATCH, 1.0),
             ("yeast", 3551, 120, 4, 5.0), ("sim350", 350, 40, 17, 2.0)]


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as exc:   # the timing stands without it, but say so
        return "nvidia-smi unavailable (%s)" % exc


def workload(name, G, H, N, DT, reps):
    torch.manual_seed(0)
    net = pb.ODENet("cuda", G, neurons=H)
    if G == bench.G and H == bench.H:
        with torch.no_grad():
            for p, src in zip(net.parameters(), bench.synthetic_weights(0, dense=False)):
                p.copy_(src.reshape(p.shape))
    gen = torch.Generator().manual_seed(1)
    y0 = torch.rand(N, 1, G, generator=gen).cuda()
    t0 = torch.rand(N, 1, generator=gen, dtype=torch.float64)
    t_rows = (t0 + torch.tensor([0.0, DT], dtype=torch.float64)).tolist()
    target = torch.rand(N, 1, G, generator=gen).cuda()
    with torch.no_grad():
        y = engine.solve_forward_many(net, y0, t_rows, True, "dopri5", 1e-7, 1e-9, 2 ** 31 - 1)
        gy = torch.zeros_like(y)
        gy[:, 1] = 2.0 * (y[:, 1] - target) / target.numel()

    def once(mask):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        engine.solve_adjoint_many(net, t_rows, True, "dopri5", 1e-7, 1e-9, 2 ** 31 - 1, y, gy, mask)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    lines = []
    with torch.no_grad():
        stats = {}
        for nm, mask in NORMS:
            pb.set_step_logging(True)
            try:
                engine.solve_adjoint_many(net, t_rows, True, "dopri5", 1e-7, 1e-9, 2 ** 31 - 1, y, gy, mask)
                logs = [pb.last_step_log(i) for i in range(N)]
                att = sum(len(x) for x in logs)
                rej = sum(1 for x in logs for s in x if not s[2])
                stats[nm] = "attempts %d, rejected %d, RHS evals / sample %.1f" % (att, rej, 2 + 6 * att / N)
            except Exception as exc:   # (the resident many-problems path logs no steps)
                stats[nm] = "steps not logged (%s)" % exc
            finally:
                pb.set_step_logging(False)
        for _, mask in NORMS:   # warm-up: module load, workspaces
            once(mask)
            once(mask)
        times = {nm: [] for nm, _ in NORMS}
        for _ in range(reps):
            for nm, mask in NORMS:
                times[nm].append(once(mask))
    base = statistics.median(times[NORMS[0][0]])
    lines.append("%s: %d x %d, %d samples, dt %g" % (name, G, H, N, DT))
    for nm, _ in NORMS:
        m = statistics.median(times[nm])
        lines.append("  %-8s median %.3f ms  min %.3f ms  max %.3f ms  (%.1f %% of default)  %s"
                     % (nm, m, min(times[nm]), max(times[nm]), 100.0 * m / base, stats[nm]))
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("seminorm_timing: needs a GPU")
    pb.set_sync_errors(True)
    lines = ["Adjoint backward, default norm vs seminorm: engine.solve_adjoint_many, CUDA events, %d alternated "
             "repetitions, all six parameters, dopri5 rtol 1e-7 / atol 1e-9" % args.reps, "card: %s" % card()]
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
