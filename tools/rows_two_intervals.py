"""Rows adjoint kernel, dopri5, one and two output intervals per problem, against the fp32 oracle run with the same norm:
relative L2 of adj_y0 and of the six parameter gradients (m, Wp, bp, Ws, bs, Wa).  5 one-row problems of 690 genes x
200 neurons (seed 11), rtol 1e-5 / atol 1e-7, loss = sum of squares of every output after the first, default norm and
seminorm.  Needs a GPU:  python tools/rows_two_intervals.py [label]"""
import os
import sys

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))
import phoenix_b200 as pb  # noqa: E402
from oracle import phoenix_oracle as O  # noqa: E402
from golden_util import rel_l2  # noqa: E402
from test_gpu_adjoint_seminorm import _problem  # noqa: E402
from test_gpu_placements import make_net  # noqa: E402
from test_gpu_time_grad import adjoint_backward_t  # noqa: E402


def main(label):
    pb.set_sync_errors(True)
    pb.engine.FORCE_ENGINE = "rows"
    rtol, atol = 1e-5, 1e-7
    for times in ((0.0, 0.1, 0.2), (0.0, 0.1)):
        w, y0, t, target = _problem(690, 200, (5, 1, 690), True, times, 11)
        net = make_net(pb, w)
        for semi in (False, True):
            net.zero_grad(set_to_none=True)
            y0g = y0.cuda().requires_grad_(True)
            opts = dict(adjoint_options={"norm": "seminorm"}) if semi else {}
            y = pb.odeint_adjoint_many(net, y0g, t, rtol=rtol, atol=atol, method="dopri5", **opts)
            ((y[:, 1:] - target.cuda()) ** 2).sum().backward()
            a_ref, g_ref = [], None
            for k in range(5):
                yr, _ = O.odeint(w, y0[k], t[k], method="dopri5", rtol=rtol, atol=atol)
                gy = torch.zeros_like(yr)
                gy[1:] = 2.0 * (yr[1:] - target[k])
                a, g, _, _ = adjoint_backward_t(w, t[k], yr, gy, "dopri5", rtol, atol, semi=semi)
                a_ref.append(a)
                g_ref = g if g_ref is None else [x + z for x, z in zip(g_ref, g)]
            errs = [rel_l2(p.grad.cpu(), r) for p, r in zip(net.parameters(), g_ref)]
            print("%-10s %-8s rows T=%d adj %.1e %s" % (label, "seminorm" if semi else "default", len(times),
                                                      rel_l2(y0g.grad.cpu(), torch.stack(a_ref)),
                                                      ["%.1e" % e for e in errs]), flush=True)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "")
