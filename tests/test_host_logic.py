"""CPU: host-side mirror of the reference interface — argument normalisation, error behaviour, module surface,
checkpoint format.  No kernels run here."""
import inspect
import os
import pickle

import pytest
import torch

import phoenix_b200 as pb
from phoenix_b200 import engine, parallel
from phoenix_b200.torchdiffeq import _api


def small_net():
    torch.manual_seed(0)
    return pb.ODENet("cpu", 30, neurons=8)


def test_module_surface_matches_reference():
    net = small_net()
    names = [n for n, _ in net.named_parameters()]
    assert names == ["gene_multipliers", "net_prods.linear_out.weight", "net_prods.linear_out.bias",
                     "net_sums.linear_out.weight", "net_sums.linear_out.bias", "net_alpha_combine.linear_out.weight"]
    assert net.gene_multipliers.shape == (1, 30)
    assert net.net_sums.linear_out.weight.shape == (8, 30)
    assert net.net_alpha_combine.linear_out.weight.shape == (30, 16)
    assert net.net_alpha_combine.linear_out.bias is None
    assert net.ndim == 30 and net.explicit_time is False
    assert "final" in inspect.getsource(pb.ODENet.forward)     # train_insilico.py:228 writes this to network.txt
    assert isinstance(net.__str__(), str)
    # init distribution of odenet.py:61-75: 95 % zeros per column, multipliers in [0, 1)
    W = net.net_sums.linear_out.weight
    assert (W == 0).float().mean() >= 0.85
    assert float(net.gene_multipliers.min()) >= 0 and float(net.gene_multipliers.max()) < 1
    assert [p is q for p, q in zip(engine.net_params(net), net.parameters())] == [True] * 6


def test_no_cpu_fallback():
    net = small_net()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        net(None, torch.rand(1, 30))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pb.odeint_adjoint(net, torch.rand(1, 30), torch.tensor([0.0, 1.0]), method="rk4")


def test_argument_errors_match_reference():
    net = small_net()
    y0, t = torch.rand(1, 30), torch.tensor([0.0, 1.0])
    with pytest.raises(ValueError, match='Invalid method "foo"'):
        pb.odeint(net, y0, t, method="foo")
    with pytest.raises(NotImplementedError):
        pb.odeint(net, y0, t, method="dopri8")
    with pytest.raises(TypeError, match="floating point"):
        pb.odeint(net, torch.zeros(1, 30, dtype=torch.long), t)
    with pytest.raises(AssertionError, match="strictly increasing or decreasing"):
        pb.odeint(net, y0, torch.tensor([0.0, 1.0, 0.5]))
    with pytest.raises(AssertionError, match="one dimensional"):
        pb.odeint(net, y0, torch.zeros(2, 2))
    with pytest.raises(ValueError, match="func must be an instance of nn.Module"):
        pb.odeint_adjoint(lambda t, y: y, y0, t)
    with pytest.raises(TypeError, match="ODENet right-hand sides only"):
        pb.odeint(torch.nn.Linear(30, 30), y0, t)


def test_odeint_adjoint_many_argument_checks():
    """The opt-in many-samples entry (SURVEY 8 f1): shape checks on the host, and no CPU fallback either."""
    net = small_net()
    y0 = torch.rand(3, 1, 30)
    t = torch.tensor([[0.0, 1.0], [0.5, 1.5], [0.2, 0.3]])
    with pytest.raises(AssertionError, match="per-sample times"):
        pb.odeint_adjoint_many(net, y0, t[0])
    with pytest.raises(AssertionError, match="same number of samples"):
        pb.odeint_adjoint_many(net, y0, t[:2])
    with pytest.raises(AssertionError, match="strictly increasing"):
        pb.odeint_adjoint_many(net, y0, torch.tensor([[0.0, 1.0], [0.5, 1.5], [0.3, 0.2]]))
    with pytest.raises(ValueError, match='Invalid method "foo"'):
        pb.odeint_adjoint_many(net, y0, t, method="foo")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pb.odeint_adjoint_many(net, y0, t, method="rk4")
    assert pb.engine._problems_per_launch(2) == 8 and pb.engine._problems_per_launch(3) == 5
    assert pb.engine._problems_per_launch(17) == 1


def test_normalise_time_handling():
    net = small_net()
    y0 = torch.rand(1, 30)
    tl, f32, rev, rtol, atol, method, mx = _api._normalise(net, y0, torch.tensor([3.0, 2.0, 0.5]), 1e-7, 1e-9, None,
                                                          None)
    assert tl == [-3.0, -2.0, -0.5] and rev and f32 and method == "dopri5" and mx == 2 ** 31 - 1
    tl, f32, rev, *_ = _api._normalise(net, y0, torch.tensor([0.0, 0.1], dtype=torch.float64), 1e-7, 1e-9, "rk4",
                                       {"max_num_steps": 5})
    assert not f32 and not rev and tl == [0.0, 0.1]


def test_flat_grad_layout_matches_reference_parameter_order():
    G, H = 7, 3
    P = 4 * G * H + 2 * H + G
    flat = torch.arange(P, dtype=torch.float32)
    views = engine.split_flat_grads(flat, G, H)
    assert [tuple(v.shape) for v in views] == [(1, G), (H, G), (H,), (H, G), (H,), (G, 2 * H)]
    assert torch.equal(torch.cat([v.reshape(-1) for v in views]), flat)


def test_checkpoint_round_trip(tmp_path, monkeypatch):
    # save() inserts the suffixes at the first '.' of the whole path, as the reference does (odenet.py:100-111), so a
    # '.' in a directory name would misplace the files: work with a bare file name inside tmp_path
    monkeypatch.chdir(tmp_path)
    net = small_net()
    fp = "model.pt"
    net.save(fp)
    for suffix in ("_prods", "_sums", "_alpha_comb", "_gene_multipliers"):
        assert os.path.exists(os.path.join(str(tmp_path), "model" + suffix + ".pt"))
    other = pb.ODENet("cpu", 30, neurons=8)
    other.load(fp)
    for a, b in zip(net.parameters(), other.parameters()):
        assert torch.equal(a, b)
    # the pickles name the activation classes through their module path, like the reference's `odenet.SoftsignMod`
    blob = pickle.dumps(net.net_sums)
    assert b"SoftsignMod" in blob


def test_shard_range_is_a_partition():
    for n in (0, 1, 7, 17, 4096):
        for w in (1, 2, 3, 8):
            spans = [parallel.shard_range(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def test_resident_plan_places_the_weight_slices():
    """phx_plan_describe (host only): where the two weight slices of a CTA live for the BASELINE shapes."""
    import ctypes
    from phoenix_b200 import _lib
    lib = _lib.load()

    def plan(G, H, B, adjoint):
        out = (ctypes.c_int32 * 8)()
        rc = lib.phx_plan_describe(148, G, H, B, adjoint, out)
        return rc, dict(zip(("ctas", "gpc", "nv", "w1", "wa", "ring_rows", "ring_stages", "smem"), list(out)))

    for adjoint in (0, 1):
        # SIM350 / SIM690 / yeast: both slices resident in shared memory, no ring
        for G, H in ((350, 40), (690, 40), (3551, 120)):
            rc, p = plan(G, H, 1, adjoint)
            assert rc == 0 and (p["w1"], p["wa"], p["ring_stages"]) == (1, 1, 0), (G, H, p)
        # breast 11165 x 200: W1 in shared memory, WA parked in tensor memory (wa == 2), nothing streams
        rc, p = plan(11165, 200, 1, adjoint)
        assert rc == 0 and (p["w1"], p["wa"], p["ring_stages"]) == (1, 2, 0), p
        assert p["ctas"] == 147 and p["gpc"] == 76 and p["nv"] == 4
        assert p["smem"] <= 227 * 1024
        # 20000 x 200: 9 rows per warp exceed the 8-row tensor-memory share -> both slices stream through the ring
        rc, p = plan(20000, 200, 1, adjoint)
        assert rc == 0 and (p["w1"], p["wa"]) == (0, 0) and p["ring_stages"] >= 1, p
    # more rows than the resident kernels take, or too many neurons: refused (the engine then streams)
    assert plan(350, 40, 9, 0)[0] != 0
    assert plan(350, 40, 5, 1)[0] != 0
    assert plan(350, 300, 1, 0)[0] != 0
    # small problems use few CTAs (cheap exchanges, room for concurrent solves): >= 16 genes per CTA, 32 from 256 genes
    rc, p = plan(37, 5, 1, 0)
    assert rc == 0 and p["ctas"] == 3 and p["gpc"] == 16
    rc, p = plan(690, 40, 1, 1)
    assert rc == 0 and p["ctas"] == 22 and p["gpc"] == 32


def test_tensor_core_work_split_covers_k_exactly():
    """phx_tc_plan_describe (host only): every K-split is a whole number of 16-k-block chunks, the splits of each half
    cover all k-blocks with no empty split, the partial-sum slots bound both halves (and the equal-cost split of the
    cotangent contractions), and the grid stays within 16 CTAs per SM (148 SMs) -- the splits come from a simulation of the
    CTA dispatch (phx_tc.cuh) -- unless the row tiles alone exceed that."""
    import ctypes
    from phoenix_b200 import _lib
    lib = _lib.load()
    out = (ctypes.c_int32 * 6)()
    for K in (1, 15, 16, 17, 350, 690, 3551, 4096, 10000, 11165, 20000):
        for M in (1, 5, 60, 128, 129, 1024, 4096, 10000, 11165, 20000):
            assert lib.phx_tc_plan_describe(K, M, out) == 0
            mtiles, ks_p, per_p, ks_s, per_s, slots = list(out)
            kb = (K + 15) // 16
            assert mtiles == (M + 127) // 128
            for ks, per in ((ks_p, per_p), (ks_s, per_s)):
                assert per % 16 == 0 and per >= 16
                assert ks >= 1 and ks * per >= kb and (ks - 1) * per < kb, (K, M, ks, per, kb)
            assert slots >= max(ks_p, ks_s) and slots <= 24
            assert mtiles * (ks_p + ks_s) <= max(16 * 148, 2 * mtiles), (K, M, list(out))
    assert lib.phx_tc_plan_describe(0, 5, out) != 0
