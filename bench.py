#!/usr/bin/env python
"""bench.py — PHOENIX NeuralODE hot path on B200: gene-steps/s (forward solve + adjoint) at the genome-scale shape.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[3], the configuration the metric "at ~11k genes" is quoted on; SURVEY.md 8d C4):
ODENet(ndim=11165, neurons=200); one step = one training-step batch of the hot path = 17 independent samples, each
`odeint_adjoint(odenet, y0[1,G], t=[tau, tau+0.0051], method='dopri5')` + MSE loss + `.backward()`
(train_insilico.py:124-140 with config_breast.cfg batch_size=17; desmedt 178-point pseudotime spacing 0.0051).
Synthetic expression values U[0,1), weights with the reference init distribution (odenet.py:61-75).

metric  gene-steps/s = B * G * (RHS evals forward + RHS-VJP evals adjoint) / time, evaluations counted by the solver.
value   device-resident inputs, C-ABI calls (phx_solve_forward_rows / phx_solve_adjoint_rows: the 17 samples of the
        step as rows of one persistent launch each, 4 in lock-step per pass, every sample its own solve with its own
        step controller; phx_unpack_grads) issued back to back.
e2e     the same step through the public Python API from pinned HOST buffers, H2D of the samples and D2H of the loss
        inside the timed region: phoenix_b200.odeint_adjoint_many (the per-sample loop of training_step as one call,
        identical solves) + backward; the literal per-sample loop over phoenix_b200.odeint_adjoint is timed beside it
        (e2e.per_sample_api_value).
N > 1   weak scaling: every rank runs its own 17 samples, then ONE NCCL sum-allreduce of the flat gradient.

--dump-outputs DIR writes what the last timed step of `value` computed as float32 DIR/<name>.npy (38 MB): y [17, 2, 1, G]
(the solution at both output times), adj_y0 [17, 1, G] (d loss / d y0) and grad_<parameter> (the six parameter gradients,
summed over the ranks).  The inputs are seeded, so two builds can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

G, H, BATCH, DT = 11165, 200, 17, 0.0051
METHOD = os.environ.get("PHX_BENCH_METHOD", "dopri5")
METRIC = "ODE RHS gene-steps/sec (fwd+adjoint) at ~11k genes"
UNIT = "gene-steps/s"
P = 4 * G * H + 2 * H + G


def synthetic_weights(seed, dense):
    """The six parameters in the reference's order (gene_multipliers, Wp, bp, Ws, bs, Wa) with its init distribution
    (odenet.py:61-75): matrices nn.init.sparse_(sparsity=0.95, std=0.05) -- per column 95 % zeros -- or dense
    N(0, 0.05^2) ("trained-like"), nn.Linear default biases, multipliers U[0,1).  Input generation only; the product arm
    never touches oracle/."""
    import math
    gen = torch.Generator().manual_seed(seed)

    def mat(rows, cols):
        w = torch.randn(rows, cols, generator=gen) * 0.05
        if not dense:
            keep = torch.rand(rows, cols, generator=gen).argsort(dim=0) >= int(math.ceil(0.95 * rows))
            w = w * keep
        return w.contiguous()

    Ws, Wp, Wa = mat(H, G), mat(H, G), mat(G, 2 * H)
    bound = 1.0 / math.sqrt(G)
    bs = (torch.rand(H, generator=gen) * 2 - 1) * bound
    bp = (torch.rand(H, generator=gen) * 2 - 1) * bound
    m = torch.rand(1, G, generator=gen)
    return [m, Wp, bp, Ws, bs, Wa]


def workload(seed, device):
    w = synthetic_weights(1003, bool(int(os.environ.get("PHX_BENCH_DENSE", "0"))))
    gen = torch.Generator().manual_seed(seed)
    y0 = torch.rand(BATCH, 1, G, generator=gen)
    target = torch.rand(BATCH, 1, G, generator=gen)
    tau = torch.rand(BATCH, generator=gen)
    t = torch.stack([tau, tau + DT], dim=1)            # [BATCH, 2] float32, like datahandler.py:107
    return w, y0, target, t


# ------------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference's torch-CPU path, all host threads
# ------------------------------------------------------------------------------------------------------------------
def cpu_sample(w, y0, target, t, n_samples):
    from oracle import phoenix_oracle as O   # the ONLY use of oracle/ in this file: the CPU baseline / reference arm
    if not isinstance(w, O.Weights):
        w = O.Weights(*w)
    evals = 0
    t0 = time.perf_counter()
    for i in range(n_samples):
        y, flog = O.odeint(w, y0[i], t[i], method=METHOD)
        gy = torch.zeros_like(y)
        gy[1] = 2.0 * (y[1] - target[i]) / target[i].numel()
        _, _, blog = O.adjoint_backward(w, t[i], y, gy, method=METHOD)
        evals += flog.nfe + blog.nfe
    dt = time.perf_counter() - t0
    return evals, dt


def cpu_prior_step(w, K, gen):
    """One prior-loss evaluation of training_step on the CPU port: prior_only_forward on K rows + its backward
    (train_insilico.py:134-138)."""
    from oracle import phoenix_oracle as O
    if not isinstance(w, O.Weights):
        w = O.Weights(*w)
    x = torch.rand(K, 1, G, generator=gen) - 0.5
    pg = torch.randn(K, 1, G, generator=gen) * 0.1
    t0 = time.perf_counter()
    J = O.rhs(w, x, decay=False)
    g = 2.0 * (J - pg) / J.numel()
    O.rhs_vjp(w, x, g, decay=False)
    return time.perf_counter() - t0


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    w, y0, target, t = workload(2000, "cpu")
    n_samples = 2
    cpu_sample(w, y0, target, t, 1)  # first call carries one-time overhead
    for _ in range(max(0, args.warmup - 1)):
        cpu_sample(w, y0, target, t, 1)
    evals, secs = 0, 0.0
    for _ in range(args.steps):
        e, s = cpu_sample(w, y0, target, t, n_samples)
        evals += e
        secs += s
    value = G * evals / secs
    sample = "%d of the %d samples of a step per timed step (fwd+adjoint, %s)" % (n_samples, BATCH, METHOD)
    line = {
        "impl": "reference", "reference_is": "CPU port of the reference (oracle/phoenix_oracle.py, pinned to the "
        "reference's own outputs by tests/golden); the reference is pure Python over torch-CPU and cannot be installed "
        "on the GPU box, see DESIGN.md section 5; timed side by side in the build container the port is ~10 % faster "
        "than the unmodified reference (profiles/r04j_port_vs_reference.txt)",
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "breast 11165 genes x 200 neurons, %s, dt=0.0051 (bounded sample)" % METHOD,
                   "genes": G, "neurons": H, "samples_per_step": n_samples},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index, rank=0):
        super().__init__(daemon=True)
        self.index, self.rank, self.rows, self.stop_flag = index, rank, [], False

    def run(self):
        # only rank 0 polls (its own GPU): an nvidia-smi process every 200 ms on each of 8 ranks is a host load the
        # end-to-end leg can see.  (In-process NVML polling was tried instead: it slows the launch path, 1.88 -> 1.90 ms.)
        if self.rank != 0:
            return
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                f = [x.strip() for x in out.stdout.strip().split(",")]
                if len(f) >= 8:
                    self.rows.append(f)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = sorted(float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for n, v in zip(names, r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        mx = max([float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()] or [0.0])
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(self.rows)}


def tensor_leg(pb, dev):
    """ODENet.forward on the synthetic-sweep shape (BASELINE config 5: 20 000 genes x 4 096 trajectories, H = 200):
    the dense branch / joint contractions on tcgen05 (3xTF32, fp32 parity).  achieved = ALGORITHMIC flops
    8*B*G*H per RHS evaluation / device time; operands (y 328 MB, weights 64 MB, f 328 MB) exceed L2."""
    Gs, Hs, Bs, reps = 20000, 200, 4096, 10
    gen = torch.Generator(device=dev).manual_seed(5)
    net = pb.ODENet(dev, Gs, neurons=Hs)
    y = torch.rand(Bs, Gs, device=dev, generator=gen)
    out = {}
    with torch.no_grad():
        for mode in ("3xtf32", "tf32"):
            pb.set_precision(mode)
            for _ in range(3):
                net(None, y)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
            ev[0].record()
            for i in range(reps):
                net(None, y)
                ev[i + 1].record()
            torch.cuda.synchronize()
            out[mode] = sum(ev[i].elapsed_time(ev[i + 1]) for i in range(reps)) / reps
    pb.set_precision("3xtf32")
    # forward + backward through autograd (ODENet.forward + the VJP for state and all six parameter cotangents):
    # 8 (forward) + 24 (VJP: recompute, state cotangent, parameter cotangents) x B*G*H algorithmic flops
    gcot = torch.randn(Bs, Gs, device=dev, generator=gen)
    def fwd_bwd():
        for p_ in net.parameters():
            p_.grad = None
        yg = y.detach().requires_grad_(True)
        net(None, yg).backward(gcot)
    for _ in range(2):
        fwd_bwd()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        fwd_bwd()
    e1.record()
    torch.cuda.synchronize()
    fb_ms = e0.elapsed_time(e1) / 5
    flops = 8.0 * Bs * Gs * Hs
    del net, y, gcot
    torch.cuda.empty_cache()
    return {"kernel": "tc_branch_kernel + tc_spfinish_kernel + tc_joint_kernel",
            "workload": "ODENet.forward, 20000 genes x 200 neurons x 4096 rows (3 launches per RHS evaluation)",
            "achieved": flops / (out["3xtf32"] * 1e-3) / 1e12, "launch_ms": out["3xtf32"],
            "algorithmic_flops": flops, "executed_mma_flops": 3.0 * flops,
            "tf32_single_pass_ms": out["tf32"], "dtype": "tf32 x3 (fp32 parity)",
            "fwd_bwd_ms": fb_ms, "fwd_bwd_achieved": 4.0 * flops / (fb_ms * 1e-3) / 1e12}


def run_ours(args):
    import torch.distributed as dist
    import phoenix_b200 as pb
    from phoenix_b200 import _lib, engine, parallel

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    w, y0_h, target_h, t_h = workload(2000 + rank, "cpu")
    net = pb.ODENet(dev, G, neurons=H)
    with torch.no_grad():
        for p, src in zip(net.parameters(), w):
            p.copy_(src)
    parallel.broadcast_parameters(net)
    lib = _lib.load()
    ctx = _lib.ctx(local)
    packed, _, _, _ = engine.packed_weights(net)
    stream = torch.cuda.current_stream(dev)
    sp = ctypes.c_void_p(stream.cuda_stream)

    # ---- device-resident leg: raw C-ABI calls --------------------------------------------------------------
    y0_d, target_d = y0_h.to(dev), target_h.to(dev)
    tl = [[float(a), float(b)] for a, b in t_h.tolist()]
    tarr = [(ctypes.c_double * 2)(*x) for x in tl]
    ws_f = torch.empty(lib.phx_rows_workspace_bytes(ctx, G, H, BATCH, 2, 0), dtype=torch.uint8, device=dev)
    ws_a = torch.empty(lib.phx_rows_workspace_bytes(ctx, G, H, BATCH, 2, 1), dtype=torch.uint8, device=dev)
    for ws in (ws_f, ws_a):   # one-time zeroing of the inter-CTA exchange area (include/phoenix_b200.h)
        _lib.check(lib.phx_solve_workspace_init(ctypes.c_void_p(ws.data_ptr()), ws.numel(), sp), "workspace_init")
    yout = torch.empty(BATCH, 2, 1, G, device=dev)
    grad_y = torch.zeros(BATCH, 2, 1, G, device=dev)
    adj_y0 = torch.empty(BATCH, 1, G, device=dev)
    nparts = lib.phx_rows_grad_parts(ctx, G, H, BATCH)
    gpk = torch.empty(nparts * lib.phx_packed_grad_bytes(G, H) // 4, device=dev)
    # N > 1: the flat gradient is written straight into a peer-mapped buffer and summed over the ranks by ONE kernel per
    # rank over NVLink peer memory (phoenix_b200/csrc/phx_peer.cu); PHX_BENCH_NCCL=1 keeps the NCCL all-reduce instead
    use_peer = world > 1 and not int(os.environ.get("PHX_BENCH_NCCL", "0"))
    peer = parallel.try_enable_peer_allreduce(net) if use_peer else None
    use_peer = peer is not None
    gsum = peer.buffer[:P] if use_peer else torch.empty(P, device=dev)
    st_f = torch.zeros(BATCH, 10, dtype=torch.int32).pin_memory()
    st_a = torch.zeros(BATCH, 10, dtype=torch.int32).pin_memory()
    mid = _lib.METHOD_IDS[METHOD]
    ptr = lambda x: ctypes.c_void_p(x.data_ptr())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    adj_ev, fwd_ev = [], []
    rows_per_pass = lib.phx_rows_supported(ctx, G, H, 1)

    # the 17 independent samples of the step go through the rows entry points: ONE persistent launch for the forward
    # solves and ONE for the adjoint sweeps, `rows_per_pass` samples in lock-step per pass, every sample its own solve with
    # its own step controller; the parameter cotangents leave the adjoint kernel already summed over the samples
    tflat = (ctypes.c_double * (2 * BATCH))(*[x for r in tl for x in r])

    def step_resident(record):
        if record:
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record(stream)
        rc = lib.phx_solve_forward_rows(ctx, G, H, BATCH, ptr(packed), ptr(y0_d), tflat, 2, 1, 0, mid, 1e-7, 1e-9,
                                        2 ** 31 - 1, ptr(yout), ptr(ws_f), ws_f.numel(), ptr(st_f), None, 0, sp)
        _lib.check(rc, "solve_forward_rows")
        if record:
            f1.record(stream)
            fwd_ev.append((f0, f1, BATCH))
        # d loss / d y(t1) for loss = mean((pred - target)^2) over the batch (train_insilico.py:132)
        _lib.check(lib.phx_mse_grad(ctx, BATCH, G, ctypes.c_void_p(yout.data_ptr() + 4 * G), 2 * G, ptr(target_d),
                                    2.0 / (BATCH * G), ctypes.c_void_p(grad_y.data_ptr() + 4 * G), 2 * G, sp), "mse_grad")
        if record:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
        rc = lib.phx_solve_adjoint_rows(ctx, G, H, BATCH, ptr(packed), tflat, 2, 1, mid, 1e-7, 1e-9, 2 ** 31 - 1,
                                        ptr(yout), ptr(grad_y), ptr(adj_y0), ptr(gpk), ptr(ws_a), ws_a.numel(),
                                        ptr(st_a), None, 0, sp)
        _lib.check(rc, "solve_adjoint_rows")
        if record:
            e1.record(stream)
            adj_ev.append((e0, e1, BATCH))
        _lib.check(lib.phx_unpack_grads(ctx, G, H, ptr(gpk), nparts, ptr(gsum), 0, sp), "unpack_grads")
        if use_peer:
            peer.reduce(numel=P)
        elif world > 1:
            dist.all_reduce(gsum)

    def timed(step_fn, steps):
        total_ms = 0.0
        for _ in range(steps):
            flush.fill_(1)                               # evict L2 between timed iterations
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            step_fn()
            b.record(stream)
            torch.cuda.synchronize()
            total_ms += a.elapsed_time(b)
        return total_ms

    for _ in range(args.warmup):
        step_resident(False)
    torch.cuda.synchronize()
    sampler = ClockSampler(local, rank)
    sampler.start()
    ms_res = timed(lambda: step_resident(True), args.steps)
    outputs = None
    if args.dump_outputs:   # copied now: the dense-weight leg below reuses these buffers
        outputs = {"y": yout, "adj_y0": adj_y0}
        for (name, _), g in zip(net.named_parameters(), engine.split_flat_grads(gsum, G, H)):
            outputs["grad_" + name.replace(".", "_")] = g
        outputs = {k: v.cpu().numpy() for k, v in outputs.items()}
    evals = 0
    for i in range(BATCH):
        evals += int(st_f[i, 3]) + int(st_a[i, 3])
        if int(st_f[i, 0]) != 0 or int(st_a[i, 0]) != 0:
            raise SystemExit("solver status non-zero: %s %s" % (st_f[i, :5].tolist(), st_a[i, :5].tolist()))
    n_attempts = sum(int(st_a[i, 1]) + int(st_a[i, 2]) for i in range(BATCH)) / BATCH
    n_vjp = sum(int(st_a[i, 3]) for i in range(BATCH)) / BATCH
    adj_ms = sum(a.elapsed_time(b) for a, b, _ in adj_ev) / sum(n for _, _, n in adj_ev)   # per sample
    fwd_ms = sum(a.elapsed_time(b) for a, b, _ in fwd_ev) / sum(n for _, _, n in fwd_ev)
    n_fwd = sum(int(st_f[i, 3]) for i in range(BATCH)) / BATCH

    # ---- end-to-end leg: reference-facing Python API from pinned host buffers ------------------------------
    y0_p, target_p = y0_h.pin_memory(), target_h.pin_memory()
    t_cpu = [t_h[i].clone() for i in range(BATCH)]
    loss_host = torch.zeros(1).pin_memory()

    def step_e2e_loop():
        # the reference's training_step verbatim: one odeint call per sample (train_insilico.py:128-130)
        net.zero_grad(set_to_none=True)
        preds = []
        tgt = target_p.to(dev, non_blocking=True)
        for i in range(BATCH):
            yb = y0_p[i].to(dev, non_blocking=True)
            preds.append(pb.odeint_adjoint(net, yb, t_cpu[i], method=METHOD)[1])
        loss = torch.mean((torch.stack(preds) - tgt) ** 2)
        loss.backward()
        if world > 1:
            parallel.allreduce_grads(net, average=False)
        loss_host.copy_(loss.detach().reshape(1), non_blocking=True)

    def step_e2e():
        # the same step with the sample loop inside the library (odeint_adjoint_many: same solves, same results)
        net.zero_grad(set_to_none=True)
        tgt = target_p.to(dev, non_blocking=True)
        yb = y0_p.to(dev, non_blocking=True)
        pred = pb.odeint_adjoint_many(net, yb, t_h, method=METHOD)[:, 1]
        loss = torch.mean((pred - tgt) ** 2)
        loss.backward()
        if world > 1:
            parallel.allreduce_grads(net, average=False)
        loss_host.copy_(loss.detach().reshape(1), non_blocking=True)

    # the per-sample loop is timed with lazy error checking (explicit opt-in: the host runs ahead of the GPU and the
    # status records are inspected at the next call / check_errors()); the default raises at the call site like the
    # reference, at the cost of one stream synchronisation per solve
    pb.set_sync_errors(False)
    for _ in range(args.warmup):
        step_e2e()
        step_e2e_loop()
    torch.cuda.synchronize()
    ms_e2e = timed(step_e2e, args.steps)
    ms_e2e_loop = timed(step_e2e_loop, max(3, args.steps // 4)) / max(3, args.steps // 4) * args.steps
    pb.check_errors()
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # ---- dense ("trained-like") weights: the same device-resident step with N(0, 0.05^2) matrices -------------------
    dense = None
    if not int(os.environ.get("PHX_BENCH_SKIP_DENSE", "0")):
        wd = synthetic_weights(1003, True)
        with torch.no_grad():
            for p_, src in zip(net.parameters(), wd):
                p_.copy_(src)
        packed, _, _, _ = engine.packed_weights(net)
        for _ in range(3):
            step_resident(False)
        torch.cuda.synchronize()
        ds = max(3, args.steps // 2)
        ms_dense = timed(lambda: step_resident(False), ds) / ds
        ev_d = sum(int(st_f[i, 3]) + int(st_a[i, 3]) for i in range(BATCH))
        dense = {"ms_per_step": ms_dense, "value_this_rank": G * ev_d / (ms_dense * 1e-3), "steps": ds,
                 "rhs_evals_per_step": ev_d, "weights": "N(0, 0.05^2) dense matrices (SURVEY 8d 'trained-like')"}
        with torch.no_grad():
            for p_, src in zip(net.parameters(), w):
                p_.copy_(src)
        packed, _, _, _ = engine.packed_weights(net)

    # ---- BASELINE metric 2: train epoch time of the breast config at N GPUs (strong scaling: the 17 samples and the
    # 10 000 prior rows of every step are split over the ranks; tools/train_epoch.py = the reference's training loop) ---
    epoch = None
    if not int(os.environ.get("PHX_BENCH_SKIP_EPOCH", "0")):
        sys.path.insert(0, os.path.join(REPO, "tools"))
        import train_epoch
        epoch = train_epoch.run_epochs("breast", epochs=2, many=True, instrument=(world == 1))
        torch.cuda.empty_cache()

    # ---- tensor-core leg (rank 0, N = 1 only; bounded): the batched RHS of BASELINE config 5 ---------------------
    tensor = None
    if rank == 0 and world == 1 and not int(os.environ.get("PHX_BENCH_SKIP_TENSOR", "0")):
        tensor = tensor_leg(pb, dev)

    # ---- reduce over ranks: time = max, work = sum -------------------------------------------------------
    stats = torch.tensor([ms_res, ms_e2e, float(evals), ms_e2e_loop], dtype=torch.float64, device=dev)
    if world > 1:
        mx = stats.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stats.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms_res, ms_e2e, evals_total, ms_e2e_loop = float(mx[0]), float(mx[1]), float(sm[2]), float(mx[3])
    else:
        evals_total = float(evals)
    work_per_step = G * evals_total                     # B = 1 per solve; evals already summed over the 17 samples
    value = work_per_step / (ms_res / args.steps / 1e3)
    e2e_value = work_per_step / (ms_e2e / args.steps / 1e3)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        # algorithmic bytes of one sample's adjoint sweep, exactly SURVEY.md 8(d): per RHS-VJP evaluation the weights
        # twice + y, a in + y', a' out (32GH + 16G bytes); per attempted step ONE 8P-byte read-modify-write of the
        # parameter cotangents.  Nothing else is counted.
        alg = n_vjp * (32.0 * G * H + 16.0 * G) + n_attempts * 8.0 * P
        achieved = alg / (adj_ms * 1e-3) / 1e9
        traffic = None
        try:
            # dram__bytes_read.sum + dram__bytes_write.sum of ONE ncu --set full capture of the 17-sample
            # phx_rows_adj_kernel launch (profiles/r02f_ncu_full.txt), per sample like achieved / algorithmic_bytes
            traffic = json.load(open(os.path.join(REPO, "profiles", "traffic.json"))).get("phx_rows_adj_kernel") / BATCH
        except Exception:
            pass
        cores = os.cpu_count() or 1
        cpu8 = cpu_epoch = None
        if world == 1:
            torch.set_num_threads(cores)
            cpu_sample(w, y0_h, target_h, t_h, 1)
            ce, cs = cpu_sample(w, y0_h, target_h, t_h, 3)
            cpu_value = G * ce / cs
            t_prior = cpu_prior_step(w, 10000, torch.Generator().manual_seed(3))
            # epoch time of the CPU port = 10 steps x (17 samples + one 10 000-row prior loss), from the timed sample
            cpu_epoch = {"epoch_s": 10 * (BATCH * cs / 3 + t_prior), "cores": cores,
                         "sample": "extrapolated from 3 samples (fwd+adjoint) and one 10 000-row prior forward+backward; "
                                   "optimiser step not included", "prior_step_s": t_prior, "sample_s": cs / 3}
            torch.set_num_threads(8)
            e8, s8 = cpu_sample(w, y0_h, target_h, t_h, 1)
            cpu8 = G * e8 / s8
            torch.set_num_threads(cores)
        else:
            cpu_value = None   # measured at N = 1 only (torchrun pins the ranks to one OpenMP thread)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "breast 11165 genes x 200 neurons, batch 17 x (odeint_adjoint %s dt=0.0051 + "
                                   "backward)" % METHOD, "genes": G, "neurons": H, "samples_per_step": BATCH,
                       "rhs_evals_per_step": evals_total / world, "l2": "flushed between timed steps (256 MiB write)",
                       "parallelism": "dp%d (samples sharded, 1 grad allreduce/step%s)" % (
                           world, "" if world == 1 else (": phx_peer_allreduce over NVLink peer memory" if use_peer
                                                         else ": NCCL"))},
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": 2 * BATCH * G * 4, "d2h_bytes_per_step": 4,
                    "api": "phoenix_b200.odeint_adjoint_many (sample loop of training_step inside the library) + "
                           "loss.backward(), pinned host inputs",
                    "per_sample_api_value": work_per_step / (ms_e2e_loop / args.steps / 1e3),
                    "per_sample_api": "phoenix_b200.odeint_adjoint once per sample, as train_insilico.py:128-130 (17 forward "
                                      "launches; the 17 adjoint nodes of the backward pass share one lock-step call)"},
            "gpu_launches": args.steps * 5,   # forward rows, loss cotangent, adjoint rows, 2 x unpack
            "roofline": {"bound": "hbm", "kernel": "phx_rows_adj_kernel", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "launch_ms": adj_ms, "algorithmic_bytes": alg,
                         "per": "one sample's adjoint sweep = the 17-sample phx_rows_adj_kernel launch / 17 (%d samples in "
                                "lock-step per pass); achieved, launch_ms, algorithmic_bytes and traffic are per sample; "
                                "algorithmic = n_vjp*(32GH+16G) + n_attempts*8P (SURVEY 8d), the weights never leave "
                                "the chip so this is algorithmic-bytes throughput, not DRAM traffic" % rows_per_pass,
                         "forward": {"kernel": "phx_rows_fwd_kernel", "launch_ms": fwd_ms,
                                     "algorithmic_bytes": n_fwd * (16.0 * G * H + 8.0 * G),
                                     "achieved": n_fwd * (16.0 * G * H + 8.0 * G) / (fwd_ms * 1e-3) / 1e9,
                                     "frac": n_fwd * (16.0 * G * H + 8.0 * G) / (fwd_ms * 1e-3) / 1e9 / peak},
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst)" if peaks else "fallback 6650"},
            "cpu_baseline": {"value": cpu_value, "unit": UNIT, "cores": cores, "kind": "port",
                             "value_8_threads": cpu8,
                             "sample": "3 of the 17 samples of one step (fwd+adjoint), after 1 warm-up sample; "
                                       "value_8_threads: 1 sample with torch.set_num_threads(8)"
                                       if world == 1 else "measured at N=1 only"},
            "clocks": sampler.summary(),
        }
        if dense is not None:
            line["dense_weights"] = dense
        if epoch is not None:
            epoch["cpu_port"] = cpu_epoch
            line["train_epoch"] = epoch
        if tensor is not None:
            bf16 = float(peaks.get("bf16_tflops", 1590.0))
            tpeak = bf16 / 2.0                            # TF32 dense = half the bf16 rate (B200_PROFILING.md)
            line["roofline_tensor"] = dict(tensor, bound="tensor", peak=tpeak, unit="TFLOP/s",
                                           frac=tensor["achieved"] / tpeak,
                                           frac_of_3xtf32_ceiling=tensor["achieved"] / (tpeak / 3.0),
                                           peak_source=("MEASURED_PEAKS.json bf16_tflops / 2" if peaks
                                                        else "fallback 1590 / 2"))
        print(json.dumps(line), flush=True)
        if outputs is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in outputs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
