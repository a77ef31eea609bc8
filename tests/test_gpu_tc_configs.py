"""The tensor-core contractions (csrc/phx_tc.cu) in every launch configuration against float64, element by element.

Every RHS call with B >= 5 rows runs four branch-type contractions on the tensor cores -- forward [S|P] (K = genes),
gSP (K = genes), Ws_bar | Wp_bar and Wa_bar (K = batch rows) -- and each is configured on the host at run time
(``branch_config`` in phx_tc.cu, reported by ``phx_tc_launch_describe``): the K split simulated by
``phx_tc_branch_plan`` (the equal-cost split for the cotangent operand), and where the A operand lives -- a ring of
4 (Hn <= 192), 3 (Hn = 208) or 2 (Hn = 224) stages in tensor memory, or shared-memory tiles (Hn = 240, 256, or a K range
shorter than two 16-k-block chunks).  The class of a contraction is (contraction, ring depth, one chunk or several per
K range, one K range or several).  ``CASES`` holds (G, H, B) shapes annotated with the class of each of their four
contractions; ``test_table_covers_every_launch_class`` (no GPU) checks that every class the library produces over the
grid below is in the table (36 classes) and that every case still lands on its classes.

Each case is compared with odenet.py:85-98 and its VJP evaluated by autograd in float64 on the GPU: f with decay, J
without, ybar and the six parameter cotangents (fresh, with PHX_VJP_REUSE_FORWARD, accumulated onto a prefilled
vector), and the fused prior loss with its cotangent and backward.  y spans [-0.25, 1.25] (warps mix the series and the
log1pf path of the log1p producers), 20 % of the multipliers are negative, and above 1 000 genes Ws and Wp are scaled by
sqrt(1000 / G) as in test_gpu_placements._inputs.

Bar on every tensor (3xTF32), met by every class: relative L2 <= 1e-5 and every element within 1e-5 * max|ref|.
Maxima observed over all cases on a B200 (148 SMs, 1000 W power limit; relative L2 / element-wise; per case and tensor
in profiles/r13a_tc_configs.txt):
  f 2.7e-6 / 3.2e-6, J 3.2e-6 / 4.2e-6, ybar 3.0e-6 / 3.4e-6, gcot 2.8e-6 / 3.8e-6, loss 4.2e-6 (relative);
  m 2.7e-6 / 3.1e-6, Wp 6.6e-6 / 8.5e-6, bp 5.0e-6 / 8.2e-6, Ws 9.0e-6 / 8.7e-6, bs 5.7e-6 / 7.5e-6, Wa 4.3e-6 / 5.2e-6.
The Ws_bar | Wp_bar sums over 10 000 rows (K = B, many chunks) come closest to the bar.  Relative L2 alone absorbs one
wrong weight row: ``test_one_wrong_row_is_rejected``.  TF32 (single pass) has its own bar TF32_L2 / TF32_ELEM
(observed <= 7.1e-4 / 7.8e-4).
"""
import collections
import ctypes
import json
import os
import subprocess
import sys

import pytest
import torch

from golden_util import rel_l2
from oracle import phoenix_oracle as O

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
SMS = 148
C_ELEM, L2_TOL = 1e-5, 1e-5
TF32_L2, TF32_ELEM = 2e-3, 2e-3
CHUNK = 16   # k-blocks per accumulation chunk (phx_tc_chunk)
NAMES = ("fwd", "gSP", "WsWp", "Wa")

Case = collections.namedtuple("Case", "G H B cls")


def C(G, H, B, *cls):
    """A (G, H, B) call; cls = (ring depth, several chunks per K range, several K ranges) of the forward [S|P], gSP,
    Ws_bar | Wp_bar and Wa_bar contractions."""
    return Case(G, H, B, tuple(cls))


CASES = [
    C(37, 1, 5, (0, 0, 0), (0, 0, 0), (0, 0, 0), (0, 0, 0)),           # everything one 16-k-block range, H = 1
    C(350, 40, 257, (0, 0, 1), (0, 0, 1), (0, 0, 1), (0, 0, 1)),       # two ranges of one chunk, ragged rows
    C(11165, 1, 5, (4, 1, 1), (4, 1, 1), (0, 0, 0), (0, 0, 0)),        # ring 4 at Hn = 16
    C(11165, 200, 5, (3, 1, 1), (3, 1, 1), (0, 0, 0), (0, 0, 0)),      # ring 3 (Hn = 208)
    C(11165, 224, 5, (2, 1, 1), (2, 1, 1), (0, 0, 0), (0, 0, 0)),      # ring 2 (Hn = 224)
    C(11165, 225, 5, (0, 1, 1), (0, 1, 1), (0, 0, 0), (0, 0, 0)),      # shared-memory A, several chunks
    C(37, 40, 10000, (0, 0, 0), (0, 0, 0), (4, 1, 1), (4, 1, 1)),      # K = B contractions on the ring
    C(37, 193, 10000, (0, 0, 0), (0, 0, 0), (3, 1, 1), (3, 1, 1)),
    C(37, 209, 10000, (0, 0, 0), (0, 0, 0), (2, 1, 1), (2, 1, 1)),
    C(37, 256, 10000, (0, 0, 0), (0, 0, 0), (0, 1, 1), (0, 1, 1)),
    C(20000, 120, 257, (4, 1, 1), (4, 1, 1), (4, 1, 0), (4, 1, 0)),    # one K range of many chunks (K = B)
    C(20000, 200, 257, (3, 1, 1), (3, 1, 1), (3, 1, 0), (3, 1, 0)),
    C(20000, 209, 257, (2, 1, 1), (2, 1, 1), (2, 1, 0), (2, 1, 0)),
    C(20000, 256, 257, (0, 1, 1), (0, 1, 1), (0, 1, 0), (0, 1, 0)),
    C(350, 100, 10000, (4, 1, 1), (4, 1, 0), (4, 1, 1), (4, 1, 1)),    # the 10 000-row prior batch
    C(350, 200, 10000, (3, 1, 1), (3, 1, 0), (3, 1, 1), (3, 1, 1)),
    C(350, 224, 10000, (2, 1, 1), (2, 1, 0), (2, 1, 1), (2, 1, 1)),
    C(350, 241, 10000, (0, 1, 1), (0, 1, 0), (0, 1, 1), (0, 1, 1)),
]
GRID_G = (37, 129, 350, 1001, 2049, 3551, 11165, 20000)
GRID_H = (1, 5, 17, 40, 100, 120, 128, 129, 176, 192, 193, 200, 208, 209, 224, 225, 240, 241, 256)
GRID_B = (5, 17, 60, 128, 129, 256, 257, 512, 513, 1024, 4096, 10000)


def _case_id(c):
    return "%dx%dxB%d" % (c.G, c.H, c.B)


def _lib():
    from phoenix_b200 import _lib as L
    return L.load()


def describe(lib, contraction, G, H, B):
    out = (ctypes.c_int32 * 8)()
    rc = lib.phx_tc_launch_describe(contraction, G, H, B, out)
    assert rc == 0, (contraction, G, H, B)
    return list(out)


def launch_class(d):
    """(ring depth, several chunks per K range, several K ranges) of a phx_tc_launch_describe record."""
    return (d[6], int(max(d[2], d[4]) > CHUNK), int(max(d[1], d[3]) > 1))


# The sweep runs in a child process: the plan cache of the library holds 64 shapes, and the grid has 192.
_SWEEP = r"""
import ctypes, json, sys
sys.path.insert(0, %r)
from phoenix_b200 import _lib as L
lib = L.load()
req = json.loads(sys.stdin.read())
out = (ctypes.c_int32 * 8)()
res = {"grid": {}, "cases": []}
def cls(c, G, H, B):
    assert lib.phx_tc_launch_describe(c, G, H, B, out) == 0
    return [out[6], int(max(out[2], out[4]) > %d), int(max(out[1], out[3]) > 1)]
for G in req["G"]:
    for H in req["H"]:
        for B in req["B"]:
            for c in range(4):
                k = json.dumps([c] + cls(c, G, H, B))
                res["grid"].setdefault(k, [G, H, B])
for G, H, B in req["cases"]:
    res["cases"].append([cls(c, G, H, B) for c in range(4)])
print(json.dumps(res))
""" % (REPO, CHUNK)


def test_table_covers_every_launch_class(monkeypatch):
    """No GPU needed: every case lands on its four classes at 148 SMs, and every class the library produces over the
    grid has a case (a planner change that creates a class or moves a case fails here, not silently on the GPU)."""
    env = {k: v for k, v in os.environ.items() if not k.startswith("PHX_TC")}
    req = {"G": GRID_G, "H": GRID_H, "B": GRID_B, "cases": [[c.G, c.H, c.B] for c in CASES]}
    res = subprocess.run([sys.executable, "-c", _SWEEP], input=json.dumps(req), capture_output=True, text=True,
                         env=env, cwd=REPO, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    res = json.loads(res.stdout)
    moved = ["%s %s: expected %s, the library launches %s" % (_case_id(c), NAMES[i], c.cls[i], tuple(got[i]))
             for c, got in zip(CASES, res["cases"]) for i in range(4) if tuple(got[i]) != c.cls[i]]
    assert not moved, "\n".join(moved)
    table = {(i,) + c.cls[i] for c in CASES for i in range(4)}
    seen = {tuple(json.loads(k)): v for k, v in res["grid"].items()}
    missing = {k: v for k, v in seen.items() if k not in table}
    assert not missing, "launch classes without a case in CASES (class: first shape): %s" % missing
    assert len(seen) == 36
    for ring in (0, 2, 3, 4):   # every A placement, with several chunks per range, on both K = G and K = B
        assert any(k[1] == ring and k[2] == 1 and k[0] == i for k in table for i in range(4))


def test_describe_follows_the_launch_rules():
    """Host-only: the ring depths of ts_plan, the two-chunk rule, the equal-cost split of the cotangent operand and of
    cached Hill planes, and argument checking."""
    lib = _lib()
    for H, ring in ((40, 4), (192, 4), (193, 3), (208, 3), (209, 2), (224, 2), (225, 0), (256, 0)):
        assert describe(lib, 0, 20000, H, 257)[6] == ring, H
    d = describe(lib, 0, 350, 40, 257)          # 22 k-blocks: shorter than two chunks -> shared-memory A
    assert d[6] == 0 and max(d[2], d[4]) < 2 * CHUNK
    g = describe(lib, 1, 20000, 120, 257)       # mode 1: equal K ranges for both halves
    assert g[1] == g[3] and g[2] == g[4]
    cached = describe(lib, 4, 20000, 120, 257)  # cached planes: the forward runs as a mode-1 launch
    assert cached[1:5] == g[1:5]
    out = (ctypes.c_int32 * 8)()
    for bad in ((5, 350, 40, 257), (8, 350, 40, 257), (-1, 350, 40, 257), (0, 350, 257, 257), (0, 0, 40, 257)):
        assert lib.phx_tc_launch_describe(*bad, out) != 0, bad


# ---- GPU ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pb():
    import phoenix_b200 as pb
    pb.set_sync_errors(True)
    yield pb
    pb.set_precision("3xtf32")


def _inputs(G, H, B, seed):
    w = O.make_weights(G, H, seed, dense=True, neg_mult_frac=0.2)
    if G > 1000:
        w.Wp.mul_((1000.0 / G) ** 0.5)
        w.Ws.mul_((1000.0 / G) ** 0.5)
    gen = torch.Generator().manual_seed(seed + 1)
    y = torch.rand(B, G, generator=gen) * 1.5 - 0.25
    g = torch.randn(B, G, generator=gen)
    pg = torch.rand(B, G, generator=gen)
    return w, y, g, pg


def _seed(c):
    return 7000 + c.G % 997 + 7 * c.H + c.B % 1013


class Rhs:
    """The RHS entry points of the C ABI on one packed copy of `w`, with a workspace of our own."""

    def __init__(self, pb, w, ws_fill=None):
        from phoenix_b200 import _lib as L, engine
        self.L, self.lib = L, L.load()
        self.G, self.H = w.G, w.H
        self.net = pb.ODENet("cuda", w.G, neurons=w.H)
        with torch.no_grad():
            for p, src in zip(self.net.parameters(), w.as_list()):
                p.copy_(src)
        self.packed = engine.packed_weights(self.net)[0]
        self.ctx = L.ctx(torch.cuda.current_device())
        self.P = 4 * w.G * w.H + 2 * w.H + w.G
        self.ws = None

    def workspace(self, B, fill=0.0):
        nb = self.lib.phx_rhs_workspace_bytes(self.G, self.H, B)
        self.ws = torch.full(((nb + 3) // 4,), fill, dtype=torch.float32, device="cuda")
        return self.ws

    def _ws(self):
        return ctypes.c_void_p(self.ws.data_ptr()), self.ws.numel() * 4

    def _st(self):
        return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def _check(self, rc, what):
        self.L.check(rc, what)
        torch.cuda.synchronize()

    def forward(self, y, B, decay):
        f = torch.empty(B, self.G, device="cuda")
        ws, nb = self._ws()
        self._check(self.lib.phx_rhs_forward(self.ctx, self.G, self.H, B, self.packed.data_ptr(), y.data_ptr(),
                                             f.data_ptr(), int(decay), ws, nb, self._st()), "rhs_forward")
        return f

    def vjp(self, y, g, B, decay, acc=0, grads=None, want_ybar=True):
        ybar = torch.empty(B, self.G, device="cuda") if want_ybar else None
        if grads is None:
            grads = torch.empty(self.P, device="cuda")
        ws, nb = self._ws()
        self._check(self.lib.phx_rhs_vjp(self.ctx, self.G, self.H, B, self.packed.data_ptr(), y.data_ptr(),
                                         g.data_ptr(), int(decay), ybar.data_ptr() if want_ybar else None,
                                         grads.data_ptr(), acc, ws, nb, self._st()), "rhs_vjp")
        return ybar, grads

    def prior_loss(self, x, pg, B):
        gcot = torch.empty(B, self.G, device="cuda")
        loss = torch.empty(1, device="cuda")
        ws, nb = self._ws()
        self._check(self.lib.phx_prior_loss(self.ctx, self.G, self.H, B, self.packed.data_ptr(), x.data_ptr(),
                                             pg.data_ptr(), ctypes.c_float(2.0 / (B * self.G)), gcot.data_ptr(),
                                             loss.data_ptr(), ws, nb, self._st()), "prior_loss")
        return loss, gcot


def split(flat, G, H):
    from phoenix_b200.engine import split_flat_grads
    return split_flat_grads(flat, G, H)


def reference(w, y, g, decay):
    """odenet.py:85-98 and its VJP by autograd in float64 on the GPU: (f, ybar, [m, Wp, bp, Ws, bs, Wa] cotangents)."""
    ps = [p.to("cuda", torch.float64).requires_grad_(True) for p in w.as_list()]
    m, Wp, bp, Ws, bs, Wa = ps
    yd = y.to("cuda", torch.float64).requires_grad_(True)
    z = yd - 0.5
    s = z / (1 + z.abs())
    l = torch.log1p(s)
    SP = torch.cat([s @ Ws.t() + bs, torch.exp(l @ Wp.t() + bp)], -1)
    f = SP @ Wa.t()
    if decay:
        f = torch.relu(m) * (f - yd)
    if g is None:
        return f.detach(), None, None
    grads = torch.autograd.grad(f, [yd] + ps, g.to("cuda", torch.float64), allow_unused=True)
    grads = [torch.zeros_like(p) if gr is None else gr for p, gr in zip([yd] + ps, grads)]
    return f.detach(), grads[0], grads[1:]


OBSERVED = collections.defaultdict(float)


def mismatches(name, a, r, c=C_ELEM, l2=L2_TOL, key=None):
    """Why `a` is not close enough to the float64 `r`: relative L2 above `l2`, or an element further than c * max|r|
    from its reference value.  Empty when it is close (an all-zero reference needs an all-zero result)."""
    a, r = a.double().reshape(-1), r.double().reshape(-1).to(a.device)
    scale = float(r.abs().max())
    if scale == 0.0:
        return [] if not a.any() else ["%s: reference is zero, result is not (max %.3e)" % (name, float(a.abs().max()))]
    rel = float((a - r).norm() / r.norm())
    emax = float((a - r).abs().max())
    ratio = emax / scale
    if key is not None:
        OBSERVED[(key, name, "l2")] = max(OBSERVED[(key, name, "l2")], rel)
        OBSERVED[(key, name, "elem")] = max(OBSERVED[(key, name, "elem")], ratio)
    print("%-10s rel_l2 %.2e  max|a-r|/max|r| %.2e" % (name, rel, ratio))
    out = []
    if not rel <= l2:
        out.append("%s: relative L2 %.3e > %.0e" % (name, rel, l2))
    if not ratio <= c:
        i = int((a - r).abs().argmax())
        out.append("%s: element %d off by %.3e (%.3e of max|ref|) > %.0e" % (name, i, float(a[i] - r[i]), ratio, c))
    return out


PNAMES = ("m", "Wp", "bp", "Ws", "bs", "Wa")


def grad_mismatches(tag, flat, ref, G, H, **kw):
    bad = []
    for n, a, r in zip(PNAMES, split(flat, G, H), ref):
        bad += mismatches("%s.%s" % (tag, n), a, r.reshape(a.shape), **kw)
    return bad


def _check_classes(pb, c):
    assert pb is not None
    lib = _lib()
    from phoenix_b200 import _lib as L
    sms = lib.phx_ctx_num_sms(L.ctx(torch.cuda.current_device()))
    assert sms == SMS, "the table is laid out for %d SMs, the device has %d" % (SMS, sms)
    got = tuple(launch_class(describe(lib, i, c.G, c.H, c.B)) for i in range(4))
    assert got == c.cls, (got, c.cls)


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=[_case_id(c) for c in CASES])
def test_case_against_float64(pb, c):
    _check_classes(pb, c)
    G, H, B = c.G, c.H, c.B
    w, y, g, pg = _inputs(G, H, B, _seed(c))
    rhs = Rhs(pb, w)
    rhs.workspace(B)
    yc, gc, pgc = y.cuda(), g.cuda(), pg.cuda()
    key = _case_id(c)
    f_ref, ybar_ref, p_ref = reference(w, y, g, True)
    J_ref, _, _ = reference(w, y, None, False)
    bad = mismatches("f", rhs.forward(yc, B, True), f_ref, key=key)
    bad += mismatches("J", rhs.forward(yc, B, False), J_ref, key=key)
    # VJP, fresh
    ybar, grads = rhs.vjp(yc, gc, B, True)
    bad += mismatches("ybar", ybar, ybar_ref, key=key)
    bad += grad_mismatches("vjp", grads, p_ref, G, H, key=key)
    # PHX_VJP_REUSE_FORWARD: the [S|P] of the forward just before is reused -- the same bits as recomputing it
    rhs.forward(yc, B, True)
    ybar2, grads2 = rhs.vjp(yc, gc, B, True, acc=2)
    assert torch.equal(ybar2, ybar) and torch.equal(grads2, grads), "the reuse path differs from the fresh one"
    # accumulate bit 0 onto a prefilled vector of the same magnitude per block
    pre = torch.cat([torch.randn(b.numel(), generator=torch.Generator().manual_seed(G + i)) * float(b.abs().max())
                     for i, b in enumerate(split(grads.cpu(), G, H))]).cuda()
    _, acc = rhs.vjp(yc, gc, B, True, acc=1, grads=pre.clone())
    bad += grad_mismatches("acc", acc.double() - pre.double(), p_ref, G, H, key=key)
    # fused prior loss, its cotangent and the backward through the reused [S|P]
    loss, gcot = rhs.prior_loss(yc, pgc, B)
    d = J_ref - pg.to("cuda", torch.float64)
    loss_ref = float((d * d).mean())
    gcot_ref = 2.0 / (B * G) * d
    rl = abs(float(loss) - loss_ref) / loss_ref
    OBSERVED[(key, "loss", "l2")] = max(OBSERVED[(key, "loss", "l2")], rl)
    if not rl <= L2_TOL:
        bad.append("loss: relative error %.3e" % rl)
    bad += mismatches("gcot", gcot, gcot_ref, key=key)
    _, pgrads = rhs.vjp(yc, gcot, B, False, acc=2, want_ybar=False)
    _, _, pp_ref = reference(w, y, gcot_ref, False)
    bad += grad_mismatches("prior", pgrads, pp_ref, G, H, key=key)
    assert not bad, "\n".join(bad)


@pytest.mark.gpu
def test_one_wrong_row_is_rejected(pb):
    """One WA row scaled by 1 + 1e-3 on the host, the float64 reference with the right weights: relative L2 of J stays
    below 1e-5, the element-wise bound rejects it.  The row is the gene whose column norm of J is closest to the
    root-mean-square column norm (a typical gene, not the largest)."""
    c = CASES[10]
    G, H, B = c.G, c.H, c.B
    w, y, _, _ = _inputs(G, H, B, _seed(c))
    J_ref, _, _ = reference(w, y, None, False)
    cols = J_ref.norm(dim=0)
    gene = int((cols - cols.pow(2).mean().sqrt()).abs().argmin())
    bad_w = O.Weights(*[p.clone() for p in w.as_list()])
    bad_w.Wa[gene] *= 1 + 1e-3
    rhs = Rhs(pb, bad_w)
    rhs.workspace(B)
    J = rhs.forward(y.cuda(), B, False)
    assert rel_l2(J.cpu(), J_ref.cpu()) < L2_TOL, "relative L2 alone should not see one row at this size"
    assert mismatches("J", J, J_ref), "one wrong WA row went unnoticed"
    assert int((J.double() - J_ref).abs().amax(0).argmax()) == gene
    ok = Rhs(pb, w)
    ok.workspace(B)
    assert not mismatches("J", ok.forward(y.cuda(), B, False), J_ref)


def _outputs(pb, c):
    """f, J, ybar, grads of case c (fresh workspace), as CPU tensors."""
    w, y, g, _ = _inputs(c.G, c.H, c.B, _seed(c))
    rhs = Rhs(pb, w)
    rhs.workspace(c.B)
    yc, gc = y.cuda(), g.cuda()
    f = rhs.forward(yc, c.B, True)
    J = rhs.forward(yc, c.B, False)
    ybar, grads = rhs.vjp(yc, gc, c.B, True)
    return {"f": f.cpu(), "J": J.cpu(), "ybar": ybar.cpu(), "grads": grads.cpu()}


def _dump(path, idx):
    import phoenix_b200 as pb
    pb.set_sync_errors(True)
    torch.save([_outputs(pb, CASES[i]) for i in idx], path)


def _child(env_extra, idx, tmp_path):
    """_outputs of CASES[idx] in a child process under extra environment variables (read once per process)."""
    path = str(tmp_path / "out.pt")
    env = dict(os.environ)
    env.update(env_extra)
    code = "import sys; sys.path[:0] = [%r, %r]; import test_gpu_tc_configs as T; T._dump(%r, %r)" % (
        HERE, REPO, path, list(idx))
    res = subprocess.run([sys.executable, "-c", code], env=env, cwd=REPO, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    return torch.load(path)


RING_CASES = [i for i, c in enumerate(CASES) if any(k[0] for k in c.cls)]
VARIANT_CASES = [4, 10, 12, 16]   # ring 2 / 4 / 2 / 2 with several chunks, K = G and K = B


@pytest.mark.gpu
def test_ts_off_is_bit_identical(pb, tmp_path):
    """PHX_TC_TS=0 keeps the A operand in shared memory: same operands, same MMA order, so every case with a ring gives
    the same bits without it."""
    theirs = _child({"PHX_TC_TS": "0"}, RING_CASES, tmp_path)
    for i, t in zip(RING_CASES, theirs):
        mine = _outputs(pb, CASES[i])
        for k in mine:
            assert torch.equal(mine[k], t[k]), (_case_id(CASES[i]), k)


@pytest.mark.gpu
def test_uv_fused_meets_the_float64_bar(pb, tmp_path):
    """PHX_TC_UV_FUSED=1: u and v of the state cotangent in the two halves of tensor memory, one pass (EMODE 3)."""
    theirs = _child({"PHX_TC_UV_FUSED": "1"}, VARIANT_CASES, tmp_path)
    bad = []
    for i, t in zip(VARIANT_CASES, theirs):
        c = CASES[i]
        w, y, g, _ = _inputs(c.G, c.H, c.B, _seed(c))
        _, ybar_ref, _ = reference(w, y, g, True)
        bad += mismatches("ybar " + _case_id(c), t["ybar"], ybar_ref.cpu(), key="uv_fused")
    assert not bad, "\n".join(bad)


@pytest.mark.gpu
def test_cta_pairs_are_bit_identical_on_multi_chunk_cases(pb):
    lib = _lib()
    for i in VARIANT_CASES:
        c = CASES[i]
        mine = _outputs(pb, c)
        lib.phx_tc_set_pair(1)
        try:
            assert all(describe(lib, k, c.G, c.H, c.B)[6] == 0 for k in range(4))
            theirs = _outputs(pb, c)
        finally:
            lib.phx_tc_set_pair(0)
        for k in mine:
            assert torch.equal(mine[k], theirs[k]), (_case_id(c), k)


@pytest.mark.gpu
@pytest.mark.parametrize("i", [10, 14], ids=lambda i: _case_id(CASES[i]))
def test_cached_hill_planes_against_float64(pb, i):
    """With cached planes the forward [S|P] (and Ws_bar | Wp_bar) run as mode-1 launches over s and l, with the
    equal-cost K split."""
    c = CASES[i]
    lib = _lib()
    plain, cached = describe(lib, 0, c.G, c.H, c.B), describe(lib, 4, c.G, c.H, c.B)
    assert launch_class(plain)[1] == 1 and launch_class(cached)[1] == 1, (plain, cached)
    assert cached[1:5] == describe(lib, 1, c.G, c.H, c.B)[1:5]
    w, y, g, _ = _inputs(c.G, c.H, c.B, _seed(c))
    rhs = Rhs(pb, w)
    rhs.workspace(c.B)
    yc, gc = y.cuda(), g.cuda()
    s, l = torch.empty_like(yc), torch.empty_like(yc)
    from phoenix_b200 import _lib as L
    L.check(lib.phx_hill_planes(rhs.ctx, yc.numel(), yc.data_ptr(), s.data_ptr(), l.data_ptr(),
                                ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), "hill_planes")
    lib.phx_hill_cache_set(rhs.ctx, yc.data_ptr(), yc.numel(), s.data_ptr(), l.data_ptr())
    try:
        J = rhs.forward(yc, c.B, False)
        _, grads = rhs.vjp(yc, gc, c.B, False, want_ybar=False)
    finally:
        lib.phx_hill_cache_set(rhs.ctx, None, 0, None, None)
    J_ref, _, p_ref = reference(w, y, g, False)
    bad = mismatches("J", J, J_ref, key="cached") + grad_mismatches("vjp", grads, p_ref, c.G, c.H, key="cached")
    assert not bad, "\n".join(bad)


@pytest.mark.gpu
@pytest.mark.parametrize("i", [2, 11, 16], ids=lambda i: _case_id(CASES[i]))
def test_tf32_mode_meets_its_own_bar(pb, i):
    c = CASES[i]
    w, y, g, _ = _inputs(c.G, c.H, c.B, _seed(c))
    rhs = Rhs(pb, w)
    rhs.workspace(c.B)
    lib = _lib()
    from phoenix_b200 import _lib as L
    lib.phx_ctx_set_precision(rhs.ctx, L.PREC_TF32)
    try:
        f = rhs.forward(y.cuda(), c.B, True)
        ybar, grads = rhs.vjp(y.cuda(), g.cuda(), c.B, True)
    finally:
        lib.phx_ctx_set_precision(rhs.ctx, L.PREC_3XTF32)
    f_ref, ybar_ref, p_ref = reference(w, y, g, True)
    kw = dict(c=TF32_ELEM, l2=TF32_L2, key="tf32")
    bad = mismatches("f", f, f_ref, **kw) + mismatches("ybar", ybar, ybar_ref, **kw)
    bad += grad_mismatches("vjp", grads, p_ref, c.G, c.H, **kw)
    assert mismatches("f", f, f_ref), "TF32 meets the 3xTF32 bar: it is not the single-pass arithmetic"
    assert not bad, "\n".join(bad)


# ---- poisoned memory -----------------------------------------------------------------------------------------------------------
def _all_outputs(rhs, y, g, pg, B, poison=None):
    """Every output of the RHS entry points on one workspace; `poison` refills the workspace before each forward."""
    def fill():
        rhs.ws.fill_(float("nan") if poison else 0.0)
    out = {}
    fill()
    out["f"] = rhs.forward(y, B, True)
    out["ybar_reuse"], out["grads_reuse"] = rhs.vjp(y, g, B, True, acc=2)
    fill()
    out["ybar"], out["grads"] = rhs.vjp(y, g, B, True)
    fill()
    out["J"] = rhs.forward(y, B, False)
    fill()
    out["loss"], out["gcot"] = rhs.prior_loss(y, pg, B)
    _, out["grads_prior"] = rhs.vjp(y, out["gcot"], B, False, acc=2, want_ybar=False)
    return {k: v.cpu() for k, v in out.items()}


def _nan_tail(x, extra):
    buf = torch.full((x.numel() + extra,), float("nan"), device="cuda")
    buf[:x.numel()] = x.reshape(-1).cuda()
    return buf


POISON_CASES = [1, 5, 10, 17]   # B % 128, G % 16 and G % 128 all non-zero; rings and shared-memory A


@pytest.mark.gpu
@pytest.mark.parametrize("i", POISON_CASES, ids=lambda i: _case_id(CASES[i]))
def test_poisoned_memory_changes_nothing(pb, i):
    """NaN directly behind the last row of y, g and prior_grad (prefixes of larger buffers), and a NaN-filled workspace
    before every forward: bit-identical outputs.  A read past B % 128, G % 16 or G % 128, or of a stale partial-sum
    slot, would bring a NaN in."""
    c = CASES[i]
    w, y, g, pg = _inputs(c.G, c.H, c.B, _seed(c))
    rhs = Rhs(pb, w)
    rhs.workspace(c.B)
    clean = _all_outputs(rhs, y.cuda(), g.cuda(), pg.cuda(), c.B)
    extra = 257 * c.G + 4096
    prefixed = _all_outputs(rhs, _nan_tail(y, extra), _nan_tail(g, extra), _nan_tail(pg, extra), c.B)
    poisoned = _all_outputs(rhs, y.cuda(), g.cuda(), pg.cuda(), c.B, poison=True)
    for k in clean:
        assert torch.isfinite(clean[k]).all(), k
        assert torch.equal(clean[k], prefixed[k]), ("NaN behind the inputs", k)
        assert torch.equal(clean[k], poisoned[k]), ("NaN-filled workspace", k)


@pytest.mark.gpu
@pytest.mark.parametrize("i", [1, 12], ids=lambda i: _case_id(CASES[i]))
def test_nan_stays_in_its_row(pb, i):
    """A NaN in one element of y: f and ybar are NaN in that row only (the other rows keep their bits) and the NaN
    pattern of every parameter cotangent is that of the float64 reference."""
    c = CASES[i]
    w, y, g, _ = _inputs(c.G, c.H, c.B, _seed(c))
    rhs = Rhs(pb, w)
    rhs.workspace(c.B)
    b0, g0 = c.B - 2, c.G - 3
    yn = y.clone()
    yn[b0, g0] = float("nan")
    f0 = rhs.forward(y.cuda(), c.B, True).cpu()
    ybar0, _ = rhs.vjp(y.cuda(), g.cuda(), c.B, True)
    f = rhs.forward(yn.cuda(), c.B, True).cpu()
    ybar, grads = rhs.vjp(yn.cuda(), g.cuda(), c.B, True)
    f_ref, ybar_ref, p_ref = reference(w, yn, g, True)
    rows = torch.arange(c.B) != b0
    for name, a, a0, r in (("f", f, f0, f_ref), ("ybar", ybar.cpu(), ybar0.cpu(), ybar_ref)):
        assert torch.equal(a[rows], a0[rows]), name
        assert torch.equal(torch.isnan(a[b0]), torch.isnan(r[b0].cpu())), name
        assert torch.isnan(a[b0]).any(), name
    for n, a, r in zip(PNAMES, split(grads.cpu(), c.G, c.H), p_ref):
        assert torch.equal(torch.isnan(a), torch.isnan(r.cpu().reshape(a.shape))), n


# ---- edge values ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("i", [1, 10, 13], ids=lambda i: _case_id(CASES[i]))
def test_huge_finite_input(pb, i):
    """One row of y at +1e38: s = 1 and l = log 2 there, as the reference and the fp32 path give (a reciprocal that
    flushes to zero would give s = l = 0).  g is scaled by 0.1 so that the multiplier cotangent sum g (J - y) stays
    finite in fp32."""
    c = CASES[i]
    w, y, g, _ = _inputs(c.G, c.H, c.B, _seed(c))
    b0 = c.B // 2
    y[b0] = 1e38
    g = 0.1 * g
    rhs = Rhs(pb, w)
    rhs.workspace(c.B)
    J = rhs.forward(y.cuda(), c.B, False)
    f = rhs.forward(y.cuda(), c.B, True)
    ybar, grads = rhs.vjp(y.cuda(), g.cuda(), c.B, True)
    J_ref, _, _ = reference(w, y, None, False)
    f_ref, ybar_ref, p_ref = reference(w, y, g, True)
    rows = torch.arange(c.B, device="cuda") != b0
    bad = mismatches("J", J, J_ref) + mismatches("f", f[rows], f_ref[rows])
    bad += mismatches("f[b0]", f[b0], f_ref[b0]) + mismatches("ybar", ybar, ybar_ref)
    bad += grad_mismatches("vjp", grads, p_ref, c.G, c.H)
    assert not bad, "\n".join(bad)


@pytest.mark.gpu
def test_tiny_multipliers_in_the_streaming_adjoint(pb):
    """Multipliers 0, 1e-30 and a subnormal (1e-40) through a streaming rk4 odeint_adjoint on B = 8 rows (the adjoint
    takes the multiplier cotangent from the RHS value it writes): the multiplier gradient against the float64 oracle."""
    G, H, B = 350, 40, 8
    w = O.make_weights(G, H, 7100, dense=True, neg_mult_frac=0.2)
    for gene, v in ((5, 0.0), (6, 1e-30), (7, 1e-40)):
        w.gene_multipliers[0, gene] = v
    assert 0 < float(w.gene_multipliers[0, 7]) < 1.2e-38
    gen = torch.Generator().manual_seed(7101)
    y0 = torch.rand(B, 1, G, generator=gen)
    target = torch.rand(1, B, 1, G, generator=gen)
    t = torch.tensor([0.0, 0.5], dtype=torch.float64)
    net = pb.ODENet("cuda", G, neurons=H)
    with torch.no_grad():
        for p, src in zip(net.parameters(), w.as_list()):
            p.copy_(src)
    saved = pb.engine.FORCE_ENGINE
    pb.engine.FORCE_ENGINE = "stream"
    try:
        y0g = y0.cuda().requires_grad_(True)
        y = pb.odeint_adjoint(net, y0g, t, method="rk4")
        torch.mean((y[1:] - target.cuda()) ** 2).backward()
    finally:
        pb.engine.FORCE_ENGINE = saved
    wd = O.Weights(*[p.double() for p in w.as_list()])
    y_ref, _ = O.odeint(wd, y0.double(), t, method="rk4")
    gy = torch.zeros_like(y_ref)
    gy[1:] = 2.0 * (y_ref[1:] - target.double()) / target.numel()
    ady, grads, _ = O.adjoint_backward(wd, t, y_ref, gy, method="rk4")
    bad = mismatches("y", y.detach(), y_ref.cuda()) + mismatches("adj_y0", y0g.grad, ady.cuda())
    m = net.gene_multipliers.grad.reshape(-1)
    bad += mismatches("m", m, grads[0].reshape(-1).cuda())
    assert float(m[5]) == 0.0
    for gene in (6, 7):
        r = float(grads[0].reshape(-1)[gene])
        assert abs(float(m[gene]) - r) <= 1e-5 * abs(r), (gene, float(m[gene]), r)
    assert not bad, "\n".join(bad)


def test_observed_maxima_are_printed():
    """(Runs last in the file under -s: prints the largest relative L2 / element-wise ratio per case and tensor.)"""
    for k in sorted(OBSERVED):
        print("%-22s %-12s %-5s %.2e" % (k[0], k[1], k[2], OBSERVED[k]))
