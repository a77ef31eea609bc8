"""Time the backward sweep of the 17-sample breast step (11 165 genes x 200 neurons, dopri5, the bench.py workload) with
the adjoint set S = all six parameters, {gene_multipliers} and {} (y0 sensitivity only).

    python tools/frozen_params_timing.py [--reps 20] [--out FILE]

One call of engine.solve_adjoint_many per timed sample (rows kernel + packed -> flat unpack), CUDA events around it; the
three sets alternate within every repetition so that they share the same clocks.  Prints the card's name and power limit
with the medians.  Needs a GPU."""
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
from phoenix_b200 import engine  # noqa: E402

SETS = [("all six", 0x3F), ("{gene_multipliers}", 0x01), ("{} (y0 only)", 0x00)]


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as exc:   # the timing stands without it, but say so
        return "nvidia-smi unavailable (%s)" % exc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("frozen_params_timing: needs a GPU")
    G, H, N, DT = bench.G, bench.H, bench.BATCH, bench.DT
    pb.set_sync_errors(True)
    net = pb.ODENet("cuda", G, neurons=H)
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

    with torch.no_grad():
        for _, mask in SETS:   # warm-up: module load, workspaces
            once(mask)
            once(mask)
        times = {name: [] for name, _ in SETS}
        for _ in range(args.reps):
            for name, mask in SETS:
                times[name].append(once(mask))
    lines = ["17-sample breast adjoint (11 165 x 200, dopri5, dt 0.0051, bench.py inputs): engine.solve_adjoint_many, "
             "rows kernel + unpack, CUDA events, %d alternated repetitions" % args.reps,
             "card: %s" % card()]
    base = statistics.median(times[SETS[0][0]])
    for name, _ in SETS:
        m = statistics.median(times[name])
        lines.append("S = %-20s median %.3f ms  min %.3f ms  max %.3f ms  (%.1f %% of all six)"
                     % (name, m, min(times[name]), max(times[name]), 100.0 * m / base))
    text = "\n".join(lines)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
