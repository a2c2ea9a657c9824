#!/usr/bin/env python
"""bench.py -- images/s of one training step (forward with batch-stat BN + RegionLoss + backward + SGD) of
yolo-pose.cfg at 416x416, batch 64 per GPU, synthetic data, random-init weights (BASELINE.json configs[1]; with
--gpus N>1 configs[2]: one process per GPU, NCCL all-reduce of the flat gradient buffer).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl ours|reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  `value` = whole-job images/s with inputs resident in HBM; `e2e` = the same step
through the reference-facing API with pinned-host inputs copied H2D and the loss read back D2H every step;
`roofline` = the tensor-core conv GEMM kernels (conv_tc2 / conv_bandt: forward + data-gradient launches) algorithmic TFLOP/s from
CUDA events recorded around every launch in an eager pass of the same steps vs the measured bf16 GEMM peak; `cpu_baseline` = the CPU oracle
port (torch-CPU restatement of the reference path) timed on this box's host cores on a bounded sample.
--impl reference times that CPU path alone (the original project has no other implementation of the hot path that runs
without a GPU).
--dump-outputs DIR writes what the last timed step computed as DIR/<name>.npy (see dump_outputs), so that two builds run with
the same arguments, hence the same seeded inputs, can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark leaves the source tree as it found it (it may be read-only)

FWD_GFLOP_PER_IMG = 29.324          # SURVEY.md 8a: 2*MAC over the 23 convs at 416x416
STEP_GFLOP_PER_IMG = 87.67          # fwd + dgrad (no dgrad for layer 0) + wgrad


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops=float(d["bf16_tflops_sustained"]), tflops_burst=float(d["bf16_tflops"]), hbm=float(d["hbm_gbs"]),
                    src="measured (MEASURED_PEAKS.json: cuBLAS bf16 sustained / copy bandwidth)")
    return dict(tflops=1400.0, tflops_burst=1590.0, hbm=6650.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def host_threads():
    """cores this process may actually use (cgroup / affinity aware), not the machine's nominal count"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


def cpu_step_factory(batch):
    """The reference's CPU path for one training step (oracle port): Darknet fwd/bwd + RegionLoss + optim.SGD."""
    import torch
    from oracle.darknet_ref import RefDarknet
    from oracle import region_loss_ref as RL
    from singleshotpose_b200 import synth
    from singleshotpose_b200.cfgs import write_cfg
    torch.manual_seed(0)
    model = RefDarknet(write_cfg()).train()
    opt = torch.optim.SGD(model.parameters(), lr=1e-4 / 64, momentum=0.9, dampening=0, weight_decay=0.0005 * 64)
    x, tgt = synth.images(batch, seed=0), synth.targets(batch, seed=1)
    # give the CPU path its best thread count: oversubscribing a big host with MKL-DNN threads is slower than using fewer
    cand = sorted({t for t in (16, 32, 64, host_threads()) if t <= host_threads()})
    best_t, best_dt = cand[-1], None
    xs = x[:2]
    for t in cand:
        torch.set_num_threads(t)
        model(xs).sum().backward()
        t0 = time.perf_counter()
        model(xs).sum().backward()
        dt = time.perf_counter() - t0
        if best_dt is None or dt < best_dt:
            best_t, best_dt = t, dt
    torch.set_num_threads(best_t)
    cpu_step_factory.threads = best_t

    def step():
        opt.zero_grad()
        out = model(x)
        loss, _ = RL.region_loss_ref(out, tgt, 20)
        loss.backward()
        opt.step()
        return float(loss)
    return step


def cpu_model_name():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def workload_config(batch, world):
    """`config` of the JSON line, identical for both arms when they run the same workload (the driver compares them)"""
    return {"workload": "train.py single-object yolo-pose.cfg, batch %d/GPU, 416x416 synthetic RGB + random 1-GT targets, "
                        "fwd(train BN)+RegionLoss(epoch 20)+bwd+SGD" % batch,
            "global_batch": batch * world, "parallelism": "dp%d" % world,
            "l2": "working set per step (>8 GB) far exceeds the 126 MB L2; no flush needed"}


DUMP_SAMPLE = 1 << 21          # sampled elements of the parameters and of their gradients: 8 MB each in float32


def dump_outputs(d, model, loss):
    """What the last timed step hands its caller: the loss it returns, and in the model it trained the parameters after the SGD
    update, their gradients and the BN running statistics.  Parameters and gradients (50.5M elements each) are sampled at fixed,
    seeded positions of the concatenation of model.parameters() in their public (OIHW) shapes, so that the sample does not depend
    on how a build lays them out in memory.  Everything is written as float32.

    The last timed step starts from the seeded initial model (main()), so its inputs are the same in every run and for every
    --steps / --warmup.  Backward kernels sum with fp32 atomics in varying order, so its outputs agree to rounding.  Measured on a
    B200 at a 1000 W power limit over runs with --steps 20, 20, 3 and 1: loss and BN statistics identical, weights within 1e-8
    and gradients within 1e-6 of their largest element, and |a - b| <= 1e-5 |a| + 1e-6 max|a| for every element."""
    import numpy as np
    import torch
    os.makedirs(d, exist_ok=True)
    params = list(model.parameters())
    total = sum(p.numel() for p in params)
    idx = torch.randint(total, (min(DUMP_SAMPLE, total),), generator=torch.Generator().manual_seed(0)).sort().values
    idx = idx.to(params[0].device)

    def cat(ts):
        return torch.cat([t.detach().reshape(-1) for t in ts])
    buffers = dict(model.named_buffers())
    out = {"loss": loss.detach().reshape(1),
           "weights": cat(params)[idx],
           "grads": cat([p.grad for p in params])[idx],
           "bn_running_mean": cat([b for n, b in buffers.items() if n.endswith("running_mean")]),
           "bn_running_var": cat([b for n, b in buffers.items() if n.endswith("running_var")])}
    for name, t in out.items():
        np.save(os.path.join(d, name + ".npy"), t.float().cpu().numpy())


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    b = args.ref_batch
    step = cpu_step_factory(b)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    v = b * args.steps / dt
    sample = "%d steps of fwd+bwd+SGD on %d synthetic 416x416 images each, torch-CPU oracle port, %d threads (%s)" % (
        args.steps, b, getattr(cpu_step_factory, "threads", host_threads()), cpu_model_name())
    print(json.dumps({
        "impl": "reference", "metric": "images/sec fwd+bwd+SGD (416x416, yolo-pose.cfg)", "value": v, "unit": "images/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(b, 1),
        "cpu_baseline": {"value": v, "unit": "images/s", "cores": getattr(cpu_step_factory, "threads", host_threads()), "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=64, help="images per GPU")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ref-batch", type=int, default=64, help="images per CPU step of the reference arm / cpu_baseline (64 = the benchmark config)")
    ap.add_argument("--buckets", type=int, default=4, help="gradient all-reduce buckets issued during backward (N > 1); 0 = one all-reduce after backward")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pnp", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time the eager launch path instead of the captured CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the loss, parameters, gradients and BN statistics of the last timed step")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from singleshotpose_b200 import Darknet, RegionLoss, FlatSGD, synth, utils
    from singleshotpose_b200.cfgs import write_cfg

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch
    torch.manual_seed(0)
    model = Darknet(write_cfg()).to(dev).train()
    init_state = {k: v.detach().clone() for k, v in model.state_dict().items()}
    crit = RegionLoss(); crit.verbose = False
    gb = B * world
    from singleshotpose_b200.optim import dp_hyperparams
    lr, wd = dp_hyperparams(0.001 * 0.1, 0.0005, B)                                          # train.py:388 + lr schedule :34-46
    opt = FlatSGD(model, lr=lr, momentum=0.9, weight_decay=wd)
    x_host = synth.images(B, seed=100 + rank).pin_memory()
    t_host = synth.targets(B, seed=200 + rank).pin_memory()
    x_dev, t_dev = x_host.to(dev), t_host.to(dev)
    eng = model._engine

    def step(x, t):
        opt.zero_grad()
        out = model(x)
        loss = crit(out, t, 20)
        loss.backward()
        if world > 1:
            opt.all_reduce_grads()
        opt.step()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    step(x_dev, t_dev)                                       # materialises the flat buffers
    if world > 1 and args.buckets > 0:
        opt.overlap_all_reduce(args.buckets)                 # SURVEY 8e: bucketed all-reduce overlapped with backward
    for _ in range(max(args.warmup, 3)):
        step(x_dev, t_dev)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # ---------------- eager pass with a CUDA-event pair around every GEMM launch (roofline of the dominant kernel) ----------------
    eng.profile = []
    l0 = eng.launches
    barrier()
    e0.record()
    for _ in range(args.steps):
        loss = step(x_dev, t_dev)
    e1.record()
    barrier()
    ms_eager = e0.elapsed_time(e1)
    launches = eng.launches - l0 + 3 * args.steps          # + RegionLoss kernel, SGD kernel is counted by the engine; zero/unpack torch ops excluded
    prof, eng.profile = eng.profile, None
    # ---------------- the product path: the whole step captured once as a CUDA graph (GraphedTrainStep) ----------------
    graphed = None
    loss = None                                              # a live autograd graph from the eager pass would pin default-stream AccumulateGrad nodes
    if not args.no_graph:
        try:
            from singleshotpose_b200 import GraphedTrainStep
            graphed = GraphedTrainStep(model, crit, opt, tuple(x_dev.shape), tuple(t_dev.shape), 20, dev, all_reduce=world > 1).capture()
        except Exception as ex:                              # capture unsupported in this configuration: stay eager, say so
            sys.stderr.write("graph capture failed (%s: %s); timing the eager path\n" % (type(ex).__name__, ex))
            graphed = None
    def eager(x, t):
        if not x.is_cuda:
            x = x_dev.copy_(x, non_blocking=True)
        return step(x, t)
    run = (lambda x, t: graphed(x, t)) if graphed is not None else eager
    for _ in range(3):
        run(x_dev, t_dev)
    # ---------------- device-resident timing (value) ----------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    e0.record()
    for _ in range(args.steps - 1):
        run(x_dev, t_dev)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    # The last timed step starts from the seeded initial model, so that what it computes is the same in every run: the steps
    # before it leave run-to-run differences (their fp32 atomics sum in varying order) that training amplifies step by step.
    # The copies go into the buffers the captured graph reads, and the conv operands are re-packed here, outside the timing.
    model.load_state_dict(init_state)
    opt._v.zero_()
    eng.pack_weights()
    barrier()
    e0.record()
    loss = run(x_dev, t_dev)
    e1.record()
    barrier()
    ms += e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model, loss)          # before the end-to-end pass trains the model further
    tmax = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms = float(tmax.item())
    value = gb * args.steps / (ms * 1e-3)
    # ---------------- end-to-end timing (host buffers) ----------------
    for _ in range(2):
        run(x_host, t_host).item()
    loss_pin = torch.empty(2, dtype=torch.float32).pin_memory()
    loss_ev = [torch.cuda.Event(), torch.cuda.Event()]
    if graphed is not None:          # warm the staged path too: its copy stream, the 133 MB staging buffer and the pinned loss buffer are
        for _ in range(2):           # created on first use and must not be billed to the timed steps (round 2: 15.06 vs 16.69 ms/step)
            graphed.stage(x_host, t_host)
            loss_pin[0].copy_(graphed.run_staged().detach().reshape(()), non_blocking=True)
        torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    e0.record()
    if graphed is not None:
        # every step: pinned host -> device copy of that step's images and targets (prefetched on a copy stream so that the PCIe
        # transfer of step i+1 overlaps the replay of step i), and the loss read back to the host
        # The loss of step i travels to a pinned host buffer right behind its replay and is READ by the host after step i+1 has been
        # enqueued (one step of software pipelining, as a training loop that logs the loss does it): every step's loss reaches the
        # host inside the timed region, the host's launch path no longer sits between two replays.
        graphed.stage(x_host, t_host)
        prev = None
        for i in range(args.steps):
            l_dev = graphed.run_staged()
            loss_pin[i & 1].copy_(l_dev.detach().reshape(()), non_blocking=True)
            loss_ev[i & 1].record()
            if i + 1 < args.steps:
                graphed.stage(x_host, t_host)
            if prev is not None:
                loss_ev[prev].synchronize(); lv = float(loss_pin[prev])
            prev = i & 1
        loss_ev[prev].synchronize(); lv = float(loss_pin[prev])
    else:
        for _ in range(args.steps):
            lv = run(x_host, t_host).item()
    e1.record()
    barrier()
    ms_e = e0.elapsed_time(e1)
    tmax = torch.tensor([ms_e], device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_e = float(tmax.item())
    e2e = gb * args.steps / (ms_e * 1e-3)

    if world > 1:
        # every rank is done with collectives here.  The captured graph holds NCCL kernels; tearing the process group
        # down underneath it can dead-lock, so the ranks synchronise once more and leave without the collective shutdown.
        dist.barrier()
        torch.cuda.synchronize()
    if rank != 0:
        sys.stdout.flush()
        os._exit(0)
    # ---------------- roofline of the dominant kernel from the per-launch events ----------------
    pk = peaks()
    agg = {}
    for kind, blk, flops, a, b in prof:
        d = agg.setdefault(kind, [0.0, 0.0, 0])
        d[0] += flops; d[1] += a.elapsed_time(b) * 1e-3; d[2] += 1
    per_kind = {k: {"tflops": v[0] / v[1] / 1e12, "ms_per_step": 1e3 * v[1] / args.steps, "launches_per_step": v[2] // args.steps}
                for k, v in agg.items() if v[1] > 0}
    # kinds: "fwd" / "dgrad" / "wgrad" = the tensor-core GEMM launches of blocks 2..31; "l0_bwd" = the CUDA-core backward of blocks 0-1
    # (csrc/l0_fused.cu: 2*N*H*W*32*27 FLOP of algebra instead of a GEMM; its forward twin is not event-timed)
    cf = agg.get("fwd", [0, 0, 0]); cd = agg.get("dgrad", [0, 0, 0])
    conv_flops, conv_t, conv_n = cf[0] + cd[0], cf[1] + cd[1], cf[2] + cd[2]
    achieved = conv_flops / conv_t / 1e12 if conv_t else 0.0
    executed = (3.0 * cf[0] + cd[0]) / conv_t / 1e12 if conv_t else 0.0     # forward launches issue 3 MMAs per algorithmic MAC
    traffic, traffic_detail = None, None
    tp = os.path.join(ROOT, "profiles", "conv_traffic.json")                 # per-launch DRAM bytes from the committed ncu --set full capture
    if os.path.exists(tp):
        try:
            traffic_detail = json.load(open(tp))
            traffic = traffic_detail["dram_bytes_read"] + traffic_detail["dram_bytes_write"]
        except Exception:
            traffic, traffic_detail = None, None
    roofline = {"bound": "tensor", "kernel": "conv GEMM launches of the forward and data-gradient passes: conv_tc2_kernel<0> (CTA pairs, N tile >= 128), "
                                             "conv_bandt_kernel (operand-swapped, N <= 64 split-fp16 / <= 128 single-term), conv_tc_kernel (the 20-channel head)", "achieved": achieved, "peak": pk["tflops"],
                "unit": "TFLOP/s", "frac": achieved / pk["tflops"], "traffic": traffic, "traffic_detail": traffic_detail, "peak_source": pk["src"],
                "executed_tflops": executed, "frac_executed": executed / pk["tflops"],
                "launches_per_step": conv_n // max(args.steps, 1), "share_of_step": conv_t / (ms_eager * 1e-3) if ms_eager else None,
                "measured_in": "separate eager pass of the same %d steps (%.2f ms/step; the graph replay that `value` times runs %.2f ms/step: "
                               "same kernels, no host launch gaps, weight-gradient GEMMs overlapped on a side stream) with an event pair around "
                               "every GEMM launch" % (args.steps, ms_eager / args.steps, ms / args.steps),
                "eager_ms_per_step": ms_eager / args.steps, "graph_ms_per_step": ms / args.steps,
                "note": "achieved/frac count ALGORITHMIC FLOPs; the forward launches execute 3 MMAs per algorithmic MAC (split-fp16 operands are "
                        "what meets the 1e-3 logits tolerance, DESIGN.md section 2), executed_tflops counts those; blocks 0-1 run in the CUDA-core l0_fused kernels (csrc/l0_fused.cu) "
                        "(HBM-bound, not part of this kernel)",
                "per_kind": per_kind,
                "step_tflops_algorithmic": STEP_GFLOP_PER_IMG * 1e9 * B / (ms / args.steps * 1e-3) / 1e12}
    # ---------------- CPU baseline (oracle port) on a bounded sample ----------------
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        nb = args.ref_batch
        cstep = cpu_step_factory(nb)
        cstep()
        t0 = time.perf_counter(); cstep(); cstep(); cstep(); dt = time.perf_counter() - t0
        cpu = {"value": 3 * nb / dt, "unit": "images/s", "cores": cpu_step_factory.threads, "kind": "port",
               "sample": "3 timed steps (after 1 warm-up) of fwd+bwd+SGD on %d synthetic 416x416 images, torch-CPU oracle, %d threads "
                         "(best of a 16/32/64/all sweep; %d usable cores), %s" % (nb, cpu_step_factory.threads, host_threads(), cpu_model_name())}
    # ---------------- PnP microbench (BASELINE.json configs[4]) ----------------
    pnp = None
    if not args.no_pnp and world == 1:
        n = 1000000
        pr = synth.pnp_problems(n, sigma=0.5, seed=5)
        P3 = torch.from_numpy(pr["P3"]).to(dev); uv = torch.from_numpy(pr["uv"]).to(dev); K = torch.from_numpy(pr["K"]).to(dev)
        utils.pnp_batched(P3, uv, K); torch.cuda.synchronize()
        e0.record(); utils.pnp_batched(P3, uv, K); e1.record(); torch.cuda.synchronize()
        tg = e0.elapsed_time(e1) * 1e-3
        pnp = {"poses_per_s": n / tg, "n": n, "points": 9, "sigma_px": 0.5, "ms": tg * 1e3}
        # achieved fp64 FLOP/s (SURVEY 8d) from the kernel's own work counters on a 64k sample: flop model of pnp_core.h per problem =
        #   4.7e3 (block assembly, one factorisation, 6 inverse iterations, the positive-definiteness proof)
        # + 1.0e3 per Rayleigh-quotient step + 1.6e4 per sweep of the 12x12 Jacobi fall-back
        # + 3.1e3 per accepted LM iteration (Jacobian, J^T J) + 5.5e2 per LM linear solve (6x6 Cholesky + reprojection error)
        from singleshotpose_b200._lib import call as _call, ptr as _ptr, stream_ptr as _sp
        ns = 65536
        Rw = torch.empty(ns, 9, dtype=torch.float64, device=dev); tw = torch.empty(ns, 3, dtype=torch.float64, device=dev)
        work = torch.zeros(ns, 3, dtype=torch.int32, device=dev)
        _call("ssp_pnp_batched_work", _ptr(P3), 1, _ptr(uv), _ptr(K), 9, ns, 20, _ptr(Rw), _ptr(tw), _ptr(work), _sp())
        w = work.cpu().numpy().astype("float64")
        rq = (-w[:, 0]).clip(min=0); sweeps = w[:, 0].clip(min=0)
        flop = 4.7e3 + 1.0e3 * rq + 1.6e4 * sweeps + 3.1e3 * w[:, 1] + 5.5e2 * w[:, 2]
        pnp["flop_per_problem_model"] = float(flop.mean())
        pnp["fp64_gflops"] = float(flop.mean()) * n / tg / 1e9
        pnp["work_mean"] = {"rq_steps": float(rq.mean()), "jacobi_fallback_fraction": float((sweeps > 0).mean()),
                            "lm_iterations": float(w[:, 1].mean()), "lm_solves": float(w[:, 2].mean())}
        pnp["bound"] = "fp64 ALU / dependent-issue latency (one problem per thread, 120 B of HBM traffic per problem)"
        try:
            import cv2
            m = 2000
            t0 = time.perf_counter()
            for i in range(m):
                _, rv, tv = cv2.solvePnP(pr["P3"], pr["uv"][i].reshape(-1, 1, 2), pr["K"], np_zeros8())
                cv2.Rodrigues(rv)
            pnp["cpu_cv2_poses_per_s"] = m / (time.perf_counter() - t0)
            pnp["cpu_sample"] = "%d problems, cv2.solvePnP loop, 1 thread" % m
        except Exception as ex:                                  # cv2 missing: baseline omitted, GPU number stands
            pnp["cpu_cv2_poses_per_s"] = None
            pnp["cpu_sample"] = "unavailable: %s" % type(ex).__name__
    # ---------------- inference path of valid.py (BASELINE.json configs[0]): eval forward + decode + PnP ----------------
    infer = None
    if world == 1 and not args.no_pnp:
        model.eval()
        P3i = torch.from_numpy(synth.box_points()).to(dev); Ki = torch.from_numpy(synth.intrinsics(np_f32())).to(dev)
        scale = torch.tensor([640.0, 480.0], device=dev)

        def infer_step(xb):
            with torch.no_grad():
                o = model(xb)
                boxes, _, _ = utils.region_boxes_batched(o, 1, 9)
                return utils.pnp_batched(P3i, boxes[:, :18].reshape(-1, 9, 2) * scale, Ki)
        infer = {}
        for bsz in (1, 64):
            xb = x_dev[:bsz]
            for _ in range(3):
                infer_step(xb)
            torch.cuda.synchronize()
            e0.record()
            reps = 20 if bsz == 1 else 5
            for _ in range(reps):
                infer_step(xb)
            e1.record(); torch.cuda.synchronize()
            msi = e0.elapsed_time(e1) / reps
            infer["batch%d" % bsz] = {"ms": msi, "images_per_s": bsz / (msi * 1e-3)}
        infer["what"] = "eval-mode forward (running-stat BN) + per-image decode + PnP, eager launches, inputs resident in HBM"
        model.train()
    # ---------------- training-image pipeline (image.py, SURVEY 8f.3): GPU vs the PIL calls of the reference ----------------
    augment = None
    if world == 1 and not args.no_pnp:
        try:
            augment = augment_extra(dev, e0, e1)
        except Exception as ex:                                  # an extra must not take the headline line down; say why
            augment = {"error": "%s: %s" % (type(ex).__name__, ex)}
    # ---------------- multi-object head (BASELINE.json configs[3]): yolo-pose-multi.cfg, batch 32 ----------------
    multi = None
    if world == 1 and not args.no_pnp:
        try:
            multi = multi_extra(dev, e0, e1)
        except Exception as ex:
            multi = {"error": "%s: %s" % (type(ex).__name__, ex)}
    out = {
        "metric": "images/sec fwd+bwd+SGD (416x416, yolo-pose.cfg)", "value": value, "unit": "images/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f16x2-split operands, f32 accumulate (fwd); f16 operands, f32 accumulate (bwd)", "data": "synthetic",
        "config": workload_config(B, world),
        "details": {"loss": lv, "launch_path": "cuda-graph replay of the whole step" if graphed is not None else "eager (ctypes launches)",
                    "grad_exchange": ("%d reverse-layer-order buckets all-reduced during backward" % args.buckets if (world > 1 and args.buckets > 0)
                                      else ("one all-reduce after backward" if world > 1 else "none (1 GPU)"))},
        "gpu_launches": launches, "clocks": clocks,
        "e2e": {"value": e2e, "unit": "images/s", "ms_per_step": ms_e / args.steps,
                "h2d_bytes_per_step": x_host.numel() * 4 + t_host.numel() * 4, "d2h_bytes_per_step": 4},
        "roofline": roofline, "cpu_baseline": cpu, "pnp": pnp, "inference": infer, "augment": augment, "multi": multi,
    }
    print(json.dumps(out))
    sys.stdout.flush()
    if world > 1:
        os._exit(0)


def augment_extra(dev, e0, e1, B=64):
    """change_background + data_augmentation + ToTensor of image.py for one training batch: 64 synthetic 640x480 LINEMOD-sized
    images + masks, 500x375 VOC-sized backgrounds -> (64,3,416,416) float32.  GPU: GpuAugmenter end to end (host byte arrays ->
    pinned staging -> one H2D copy -> kernels), CUDA events.  CPU: the same PIL calls the reference makes, 1 thread, 8 samples."""
    import random
    import numpy as np
    import torch
    from singleshotpose_b200 import image as I, synth
    samples = [synth.photo_sample(i) for i in range(8)]
    imgs, masks, bgs = [[s[k] for s in samples] * (B // 8) for k in range(3)]
    aug = I.GpuAugmenter(dev)
    rng = random.Random(0)
    for _ in range(3):
        x, params = aug(imgs, masks, bgs, (416, 416), rng=rng)
    torch.cuda.synchronize()
    reps = 5
    t0 = time.perf_counter()
    e0.record()
    for _ in range(reps):
        x, params = aug(imgs, masks, bgs, (416, 416), rng=rng)
    e1.record(); torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / reps
    ms = e0.elapsed_time(e1) / reps
    res = {"images_per_s": B / wall, "ms_per_batch_wall": wall * 1e3, "ms_per_batch_device_span": ms, "batch": B,
           "h2d_bytes_per_batch": aug.h2d_bytes, "out_bytes_per_batch": x.numel() * 4,
           "what": "64 x (640x480 image+mask, 500x375 background) -> 416x416 float32, BICUBIC (Pillow's resize() default), "
                   "wall time includes host staging (numpy copies into pinned memory, point() tables) and the H2D copy"}
    try:
        from PIL import Image
        lp, ln = I.mask_luts()
        m = 8
        t0 = time.perf_counter()
        for i in range(m):
            p = params[i]
            im, mk, bg = (Image.fromarray(a) for a in samples[i])
            bgr = np.asarray(bg.resize(im.size))
            comp = np.clip(np.asarray(im).astype(np.int32) * lp[np.asarray(mk)] + bgr.astype(np.int32) * ln[np.asarray(mk)], 0, 255).astype(np.uint8)
            c = Image.fromarray(comp).crop((p["pleft"], p["ptop"], p["pleft"] + p["cw"], p["ptop"] + p["ch"])).resize((416, 416))
            h, s, v = c.convert("HSV").split()
            lh, ls, lv = I.distort_luts(p["dhue"], p["dsat"], p["dexp"])
            c = Image.merge("HSV", (h.point(list(lh)), s.point(list(ls)), v.point(list(lv)))).convert("RGB")
            ref = torch.from_numpy(np.asarray(c).copy()).permute(2, 0, 1).float().div(255)
        res["cpu_pil_images_per_s"] = m / (time.perf_counter() - t0)
        res["cpu_sample"] = "%d samples, the PIL calls of image.py (resize/crop/convert/point/merge), 1 thread; the numpy mask blend stands in for ImageMath" % m
        res["last_sample_identical_to_pil"] = bool(torch.equal(ref, x[m - 1].cpu()))
    except Exception as ex:
        res["cpu_pil_images_per_s"] = None
        res["cpu_sample"] = "unavailable: %s" % type(ex).__name__
    return res


def multi_extra(dev, e0, e1, B=32):
    """configs[3]: yolo-pose-multi.cfg at batch 32 -- eval forward + get_multi_region_boxes (conf_thresh 0.05), and the training
    step's forward + RegionLoss-multi + backward (1-3 GTs per image)."""
    import torch
    from singleshotpose_b200 import synth
    from singleshotpose_b200.cfgs import write_cfg
    from singleshotpose_b200.darknet_multi import Darknet as DarknetMulti
    from singleshotpose_b200.region_loss_multi import RegionLoss as RegionLossMulti
    from singleshotpose_b200.utils_multi import get_multi_region_boxes
    torch.manual_seed(0)
    m = DarknetMulti(write_cfg(multi=True)).to(dev)
    x = synth.images(B, seed=3).to(dev)
    tgt = synth.targets_multi(B, seed=5)
    crit = RegionLossMulti(anchors=m.anchors); crit.verbose = False
    res = {}
    m.train()
    for _ in range(3):
        for p in m.parameters():
            p.grad = None
        crit(m(x), tgt, 20).backward()
    torch.cuda.synchronize()
    reps = 5
    e0.record()
    for _ in range(reps):
        for p in m.parameters():
            p.grad = None
        loss = crit(m(x), tgt, 20)
        loss.backward()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    res["train_fwd_loss_bwd"] = {"ms": ms, "images_per_s": B / (ms * 1e-3), "loss": float(loss.detach())}
    m.eval()
    with torch.no_grad():
        for _ in range(2):
            get_multi_region_boxes(m(x), 0.05, 13, 9, m.anchors, 5, 3, only_objectness=0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            boxes = get_multi_region_boxes(m(x), 0.05, 13, 9, m.anchors, 5, 3, only_objectness=0)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / reps
    res["eval_fwd_decode"] = {"ms": dt * 1e3, "images_per_s": B / dt, "boxes": int(sum(len(b) for b in boxes))}
    res["what"] = "yolo-pose-multi.cfg, batch %d, 416x416 synthetic, eager launches; decode returns the reference's python box lists (wall clock)" % B
    return res


def np_f32():
    import numpy as np
    return np.float32


def np_zeros8():
    import numpy as np
    return np.zeros((8, 1), np.float32)


if __name__ == "__main__":
    main()
