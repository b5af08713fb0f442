#!/usr/bin/env python
"""Benchmark of the Ladder-VAE hot path (BASELINE.json metric: train images/s, CIFAR10 15-layer LVAE,
batch 256 per GPU, data-parallel over N B200s).

    python bench.py --gpus N --steps K --warmup W              # our sm_100a path
    python bench.py --impl reference --gpus N --steps K ...    # the reference's CPU path (oracle port)
    python bench.py --workload iw ...                          # IW-1000 evals/s on the 12-layer MNIST model
    python bench.py ... --dump-outputs DIR                     # also write the last timed step's outputs as DIR/*.npy

For N > 1 launch with torch.distributed.run (one rank per GPU).  Rank 0 prints ONE JSON line, last.
A "step" is one ELBO training step (zero grads, forward, loss, backward, gradient all-reduce,
Adamax) over one synthetic batch.  `value` is timed with the batch already resident in HBM;
`e2e` is timed through the public TrainEngine.step(x_host) call with the pinned-host -> device
copy of the batch and the device -> host read of the loss inside the timed region.

The default (train) line also carries the rest of BASELINE.json's metric and configs as sub-records, each timed the same
way (warm-up, barrier, CUDA events, max over ranks): `iw` = the IW-1000 bound on the 12-layer MNIST model with the samples
sharded over the N ranks (the second half of the metric), `configs` = one short timing each of the MNIST-3 / MNIST-12 /
CelebA-20 training steps, `value_f32` = the headline step in the exact-fp32 parity mode, `dp_check` (N > 1) = replicas
hold bit-identical parameters after the timed steps and the NCCL-reduced gradient arena equals the sum of the per-rank
gradients.  `--no-extras` skips them (A/B timing runs).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CONFIGS = {"train": ("cifar15", 256), "iw": ("mnist12", 1000), "mnist12": ("mnist12", 128), "mnist3": ("mnist3", 64),
           "celeba20": ("celeba20", 64)}
# algorithmic conv GFLOP per image, forward / total (SURVEY.md section 8)
CONV_GFLOP = {"mnist3": (1.042, 3.126), "mnist12": (2.913, 8.737), "cifar15": (3.655, 10.962), "celeba20": (14.759, 44.266)}
METRIC_NAME = {"cifar15": "CIFAR10 15-layer", "mnist3": "MNIST 3-layer", "mnist12": "MNIST 12-layer", "celeba20": "CelebA 20-layer"}
CPU_BATCH = 32          # the CPU arms time a bounded sample: steps of this batch (CPU throughput is flat in the batch size)


def train_config(cfg_name, batch, world, graph):
    """`config` of a training line -- printed identically by our arm and by the reference arm."""
    lik = "Bernoulli" if cfg_name.startswith("mnist") else "10-component DMoL"
    return {"workload": "ELBO training step (zero grad, forward, loss, backward, gradient all-reduce, Adamax), "
                        "%s, %s, dropout 0.2, train-mode BatchNorm" % (cfg_name, lik),
            "per_gpu_batch": batch, "global_batch": batch * world, "parallelism": "dp%d" % world,
            "precision": "GPU arm: bf16 activations + tcgen05 convolutions with fp32 accumulation, fp32 stochastic / likelihood "
                         "parameters, fp32 master weights (value_f32 = the exact-fp32 mode); reference arm: fp32 on the host CPU",
            "reference_arm_sample": "the CPU arm times steps of batch %d, not %d (a bounded sample; CPU throughput is flat in "
                                    "the batch size)" % (CPU_BATCH, batch),
            "cuda_graph": graph,
            "l2_policy": "inputs larger than L2: a step streams several GB of activations (peak_mem_gb)"}


def iw_config(K, world, batch, full_forward):
    return {"workload": "importance-weighted bound, K=%d samples sharded over %d GPU(s), test batch %d, "
                        "binarized-MNIST-shaped 12-layer LVAE, eval mode" % (K, world, batch),
            "bottom_up_pass": "per sample (as the reference)" if full_forward else "once per image batch (eval mode is deterministic)",
            "reference_arm_sample": "the CPU arm times eval-mode forwards of batch 32 and extrapolates to K = %d" % K,
            "l2_policy": "per-sample working set exceeds L2"}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


def synthetic_batch(cfg, batch, seed):
    """SURVEY.md 8d: Bernoulli(0.15) binary images or uint8-grid uniform RGB, numpy seeded."""
    import numpy as np
    import torch
    rng = np.random.RandomState(seed)
    shp = (batch, cfg.color_ch) + tuple(cfg.img_shape)
    if cfg.likelihood_form == "bernoulli":
        x = (rng.random_sample(shp) < 0.15).astype(np.float32)
    else:
        x = rng.randint(0, 256, size=shp).astype(np.float32) / 255.0
    return torch.from_numpy(x)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.proc, self.path = gpu_index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:  # noqa: BLE001
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for line in open(self.path):
            f = [t.strip() for t in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_baseline_train(cfg_name, cpu_batch, steps, warmup=1):
    """The reference's CPU path (oracle port, same op sequence in PyTorch CPU ops) on a bounded sample."""
    import torch
    from oracle import lvae_oracle as O
    cfg = O.baseline_config(cfg_name)
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(42)
    st = O.TrainState(cfg, O.make_params(cfg, 42))
    x = synthetic_batch(cfg, cpu_batch, 0)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        st.step(x)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    t = statistics.median(times)
    return dict(value=cpu_batch / t, unit="images/s", cores=torch.get_num_threads(), kind="port",
                sample="%d training steps of batch %d (same model, fp32, torch CPU ops via the oracle port), median"
                       % (steps, cpu_batch), s_per_step=t)


def cpu_baseline_iw(cpu_batch, forwards):
    import torch
    from oracle import lvae_oracle as O
    cfg = O.baseline_config("mnist12")
    torch.set_num_threads(os.cpu_count() or 1)
    P = O.make_params(cfg, 42)
    x = synthetic_batch(cfg, cpu_batch, 0)
    times = []
    with torch.no_grad():
        for i in range(1 + forwards):
            t0 = time.perf_counter()
            O.forward(P, cfg, x, None, None, False)
            if i >= 1:
                times.append(time.perf_counter() - t0)
    t = statistics.median(times)
    return dict(value=cpu_batch / t / 1000.0, unit="images/s with a 1000-sample bound", cores=torch.get_num_threads(), kind="port",
                sample="%d eval-mode forwards of batch %d, extrapolated to K=1000 (the reference recomputes the full "
                       "forward per sample)" % (forwards, cpu_batch), s_per_forward=t)


def run_reference(args, rank):
    if rank != 0:
        return
    name, batch = CONFIGS[args.workload]
    t0 = time.perf_counter()
    if args.workload == "iw":
        cb = cpu_baseline_iw(32, max(1, args.steps))
        metric, unit = "IW-1000 evals/s (MNIST 12-layer LVAE)", "images/s with a 1000-sample bound"   # = our arm's
        cfgd = iw_config(1000, args.gpus, batch, False)
        ms = cb["s_per_forward"] * 1e3
    else:
        cb = cpu_baseline_train(name, CPU_BATCH, max(1, args.steps), max(1, min(args.warmup, 1)))
        metric, unit = "train images/s (%s LVAE)" % METRIC_NAME.get(name, name), "images/s"
        cfgd = train_config(name, batch, args.gpus, True)           # the same dict our arm prints
        ms = cb["s_per_step"] * 1e3
    line = {"impl": "reference", "metric": metric, "value": cb["value"], "unit": unit, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong" if args.workload == "iw" else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfgd,
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t0}
    print(json.dumps(line), flush=True)


def conv_roofline(torch, pk, dtype="bf16"):
    """Dominant kernel: 3x3 64->64 stride-1 conv (335 of 538 forward convs, SURVEY.md 2a) at the most
    common CIFAR-15 shape (B=256, 16x16).  Timed alone with CUDA events on the launch stream over
    rotating buffers larger than L2; the launches are replayed from a CUDA graph (as in the step), so that the host-side
    tensor-map encodes of an eager launch loop are not inside the timed region."""
    from lvae_b200 import _capi, ops
    B, H, W, C, k = 256, 16, 16, 64, 3
    tdt = torch.bfloat16 if dtype == "bf16" else torch.float32
    nbuf = 12 if dtype == "bf16" else 6             # (in + out) x nbuf > 126 MB L2
    xs = [torch.randn(B, H, W, C, device="cuda").to(tdt) for _ in range(nbuf)]
    ys = [torch.empty(B, H, W, C, device="cuda", dtype=tdt) for _ in range(nbuf)]
    bias = torch.zeros(C, device="cuda")
    w = torch.randn(C, C, k, k, device="cuda") / 24.0
    if dtype == "bf16":
        pack = ops.WeightPack(C, C, k * k, 2)
        wp = pack.get(w, torch.bfloat16)
        name = "conv_tc_kernel 3x3 64->64 B=256 16x16 (TMA + tcgen05.mma + TMEM, bf16 in / fp32 accumulate)"

        def launch(i):
            _capi.call("lvae_conv2d_tc", xs[i % nbuf].data_ptr(), None, wp.data_ptr(), bias.data_ptr(), None, None,
                       ys[i % nbuf].data_ptr(), None, 0, B, H, W, C, C, k, 0, 0, torch.cuda.current_stream().cuda_stream)
    else:
        pack = ops.WeightPack(C, C, k * k, 0)
        wp = pack.get(w, torch.float32)
        name = "conv_gather_kernel<float> 3x3 64->64 B=256 16x16 (fp32 CUDA-core implicit GEMM)"

        def launch(i):
            _capi.call("lvae_conv2d_gather", xs[i % nbuf].data_ptr(), None, wp.data_ptr(), bias.data_ptr(), None, None, None,
                       ys[i % nbuf].data_ptr(), B, H, W, C, 0, H, W, C, C, k, k, 1, 1, 0, 0, torch.cuda.current_stream().cuda_stream)
    for i in range(5):
        launch(i)
    torch.cuda.synchronize()
    n, reps = 48, 4
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(n):
            launch(i)
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / (n * reps)
    flops = 2.0 * B * H * W * C * C * k * k
    achieved = flops / (us * 1e-6) / 1e12
    bytes_alg = 2.0 * B * H * W * C * (2 if dtype == "bf16" else 4)
    return {"bound": "tensor", "kernel": name, "achieved": achieved, "peak": pk["tf_burst"], "unit": "TFLOP/s",
            "frac": achieved / pk["tf_burst"], "traffic": NCU_CONV_DRAM_BYTES if dtype == "bf16" else None,
            "traffic_unit": "bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum, profiles/ncu_conv_tc_r01_final.txt)",
            "us_per_launch": us, "flops_per_launch": flops,
            "algorithmic_bytes_per_launch": bytes_alg, "hbm_gbs_at_this_rate": bytes_alg / (us * 1e-6) / 1e9,
            "peak_source": "%s bf16 burst (kernel timed alone)" % pk["src"],
            "timing": "CUDA-graph replay of %d launches x %d, CUDA events on the replay stream" % (n, reps),
            "shape_limit": "the layer width is the reference's: an M=128, N=64, K=16 SS-mode tcgen05.mma needs 32 tensor cycles "
                           "but reads 6 KB of shared-memory operands = 48 cycles of the 128 B/clk port (57 measured), so "
                           "<= 2/3 of the peak at best; 512 tiles on 148 CTAs add a 4-vs-3.46 wave quantisation"}


def hbm_rooflines(workload):
    """Secondary roofline entries for the HBM-bound kernels north_star names (fused stochastic block, likelihoods): the
    microbenchmarks of profiles/bench_hbm_kernels.py (CUDA-graph replay over rotating buffers larger than L2, CUDA events on
    the capturing stream, algorithmic bytes of SURVEY.md 8d over the measured copy bandwidth).  Never fatal: an exception
    is reported in place of the numbers; the table it prints goes to stderr."""
    import contextlib
    import importlib.util
    try:
        spec = importlib.util.spec_from_file_location("bench_hbm_kernels", os.path.join(ROOT, "profiles", "bench_hbm_kernels.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        peak, src = mod.hbm_peak()
        rows = []
        with contextlib.redirect_stdout(sys.stderr):
            if workload == "iw":
                mod.bench_stochastic(rows, peak, src, B=1000)
                mod.bench_bernoulli(rows, peak, src)
            else:
                mod.bench_stochastic(rows, peak, src)
                mod.bench_dmol(rows, peak, src)
        keep = ("kernel", "shape", "us_per_launch", "achieved", "peak", "unit", "frac", "bound")
        return [{k: r[k] for k in keep} for r in rows]
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)[:300]}


# dram__bytes_read.sum + dram__bytes_write.sum of this kernel from one `ncu --set full` capture (profiles/ncu_conv_tc_r01_final.txt):
# 8.53 MB read (8.39 MB activations + weights), 0 written (the output is still dirty in L2 when the kernel ends)
NCU_CONV_DRAM_BYTES = 8526336


class Ctx:
    """Rank / world plumbing shared by the timed sections."""

    def __init__(self, torch, dist, rank, world, local):
        self.torch, self.dist, self.rank, self.world, self.local = torch, dist, rank, world, local

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v):
        if self.world == 1:
            return v
        t = self.torch.tensor([v], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t)


def kernel_shares(torch, engine):
    """CUPTI (torch.profiler) over ONE replayed step: device time per kernel family.  Not a timing of record (profiler
    attached) -- it only apportions the step, which is timed separately, to kernel families."""
    import collections
    try:
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            engine.step(None)
            torch.cuda.synchronize()
        agg = collections.defaultdict(lambda: [0, 0.0])
        for e in prof.events():
            if e.device_type != torch.autograd.DeviceType.CUDA:
                continue
            name = e.name.replace("(anonymous namespace)::", "").split("(")[0].split("<")[0].strip()
            if name.startswith("void "):
                name = name[5:]
            if name.startswith("at::"):
                name = "aten_glue"
            elif "nccl" in name.lower():
                name = "nccl"
            elif name.startswith("Memset") or name.startswith("Memcpy"):
                name = "memset_memcpy"
            agg[name][0] += 1
            agg[name][1] += (e.time_range.end - e.time_range.start)
        return {k: {"launches": v[0], "us": round(v[1], 1)} for k, v in sorted(agg.items(), key=lambda kv: -kv[1][1])}
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)[:200]}


DUMP_SAMPLE = 1 << 20      # entries kept of each dumped array larger than this (a fixed, seeded choice)


def dump_outputs(path, arrays):
    """Write each array as <path>/<name>.npy (float64).  An array of more than DUMP_SAMPLE entries is replaced by the same
    seeded sample of its flattened entries in every run, so that two builds can be compared output for output."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        if a.size > DUMP_SAMPLE:
            a = a.reshape(-1)[np.sort(np.random.RandomState(0).choice(a.size, DUMP_SAMPLE, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


def train_step_outputs(model, out):
    """What a caller of TrainEngine.step holds after a step: the returned scalars, and the model's updated parameters,
    their gradients and the BatchNorm running statistics (in the model's own parameter / buffer order)."""
    import torch
    params = [p for p in model.parameters() if p.requires_grad]
    res = {k: v.detach().double().cpu().numpy() for k, v in out.items()}
    res["params"] = torch.cat([p.detach().flatten() for p in params]).cpu().numpy()
    res["grads"] = torch.cat([p.grad.detach().flatten() for p in params]).cpu().numpy()
    res["buffers"] = torch.cat([b.detach().double().flatten() for b in model.buffers()]).cpu().numpy()
    return res


def time_train(cx, cfg_name, batch, dtype, steps, warmup, graph=True, side_streams=3, with_e2e=True, sampler=None,
               shares=False, dp_check=False, dump=None):
    """Build the model, warm up, time `steps` steps device-resident (`value`) and through TrainEngine.step(x_host) (`e2e`).
    `dump`: directory that receives what the last device-resident timed step computed (rank 0)."""
    torch = cx.torch
    import lvae_b200
    from lvae_b200.engine import TrainEngine
    from lvae_b200.configs import baseline_config
    cfg = baseline_config(cfg_name)
    torch.manual_seed(42)
    lvae_b200.manual_seed(1234)             # the engine folds the rank into the Philox key
    model = lvae_b200.LadderVAE(**cfg.kwargs()).cuda()
    if dtype == "bf16":
        model.set_compute_dtype(torch.bfloat16)
    x_host = synthetic_batch(cfg, batch, cx.rank).pin_memory()
    engine = TrainEngine(model, batch, use_graph=graph, wgrad_side_stream=side_streams)
    torch.cuda.reset_peak_memory_stats()
    for _ in range(warmup):
        engine.step(x_host)
    torch.cuda.synchronize()
    mem_gb = torch.cuda.max_memory_allocated() / 2 ** 30
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cx.barrier()
    if sampler is not None:
        sampler.start()
    e0.record()
    for _ in range(steps):
        out = engine.step(None)
    e1.record()
    cx.barrier()
    clocks = sampler.stop() if sampler is not None else None
    ms = cx.max_over_ranks(e0.elapsed_time(e1)) / steps
    if dump and cx.rank == 0:
        dump_outputs(dump, train_step_outputs(model, out))
    res = {"value": batch * cx.world / (ms * 1e-3), "unit": "images/s", "ms_per_step": ms, "steps": steps, "warmup": warmup,
           "dtype": dtype, "per_gpu_batch": batch, "launches_per_step": engine.launches_per_step, "peak_mem_gb": mem_gb,
           "loss": float(out["loss"]), "clocks": clocks}
    gflop = CONV_GFLOP[cfg_name][1]
    res["conv_tflops_per_gpu"] = res["value"] / cx.world * gflop / 1e3
    if with_e2e:
        loss_host = torch.zeros((), dtype=torch.float32).pin_memory()
        cx.barrier()
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            out = engine.step(x_host)                         # pinned host -> device copy inside
            loss_host.copy_(out["loss"], non_blocking=False)  # device -> host read of the loss
        e1.record()
        cx.barrier()
        e2e_ms = cx.max_over_ranks(e0.elapsed_time(e1)) / steps
        res["e2e"] = {"value": batch * cx.world / (e2e_ms * 1e-3), "unit": "images/s", "h2d_bytes_per_step": x_host.numel() * 4,
                      "d2h_bytes_per_step": 4, "wall_ms_per_step": (time.perf_counter() - t0) * 1e3 / steps}
    if shares and cx.rank == 0:
        res["kernel_shares"] = kernel_shares(torch, engine)
    elif shares:
        engine.step(None)                   # keep the ranks in lock-step (the all-reduce inside the step is a collective)
    if dp_check and cx.world > 1:
        res["dp_check"] = run_dp_check(cx, engine)
    engine.arena.detach_sinks()
    del engine, model
    torch.cuda.empty_cache()
    return res


def run_dp_check(cx, engine):
    """(1) After the timed steps every replica must hold bit-identical parameters (same reduced gradients, same Adamax);
    (2) one more forward/backward: the NCCL-reduced gradient arena must equal the sum of the per-rank arenas (gathered and
    summed in fp64 here)."""
    torch, dist = cx.torch, cx.dist
    flat = engine.arena.flat
    ref0 = flat.clone()
    dist.broadcast(ref0, 0)                                   # rank 0's parameters
    d = torch.stack([(flat - ref0).abs().max().double(), (flat.view(torch.int32) != ref0.view(torch.int32)).sum().double()])
    dist.all_reduce(d, op=dist.ReduceOp.MAX)
    param_diff, param_bits = float(d[0]), int(d[1])
    where = []
    if param_bits and cx.rank == cx.world - 1:                # which tensors (diagnostic; printed to stderr by the last rank)
        names = {id(p): n for n, p in engine.model.named_parameters()}
        bad = (flat.view(torch.int32) != ref0.view(torch.int32))
        for p in engine.arena.params:
            off = engine.arena.offsets[id(p)]
            c = int(bad[off:off + p.numel()].sum())
            if c:
                where.append((c, p.numel(), names[id(p)], engine._bucket_of[id(p)]))
        where.sort(reverse=True)
        sys.stderr.write("dp_check: %d tensors with elements that differ from rank 0; largest: %s\n" % (len(where), where[:12]))
    # gradient arena: the engine's (overlapped, bucketed) NCCL reduction against a manual fp64 sum of the per-rank arenas.
    # Pass 1 with the reduction switched off gives this rank's own gradients; pass 2 replays the same step (same Philox
    # state) through the engine's normal path.
    from lvae_b200 import ops
    rng = ops.rng_state(torch.device("cuda", torch.cuda.current_device()))
    rng0 = rng.clone()
    overlap = engine.overlap
    engine.overlap = False
    engine._forward_backward()
    torch.cuda.synchronize()
    g_local = engine.arena.grad.clone()
    n = g_local.numel()
    chunk = torch.empty((cx.world, n), dtype=torch.float32, device="cuda")
    dist.all_gather_into_tensor(chunk, g_local)
    manual = chunk.double().sum(0)
    engine.overlap = overlap
    rng.copy_(rng0)
    engine._forward_backward()
    engine._all_reduce()
    torch.cuda.synchronize()
    red = engine.arena.grad.double()
    gdiff = float((red - manual).abs().max() / manual.abs().max())
    gdiff_l2 = float((red - manual).norm() / manual.norm())
    # per bucket, against the bucket's own largest gradient (a bucket reduced too early shows up here even if its
    # gradients are small next to the global maximum)
    gdiff_bucket = max(float((red[s:e] - manual[s:e]).abs().max() / manual[s:e].abs().max().clamp_min(1e-30)) for s, e in engine.buckets)
    # how different the per-rank gradients were (a check that the ranks really saw different data / noise)
    spread = float((chunk[0].double() - manual / cx.world).abs().max() / manual.abs().max() * cx.world)
    return {"param_max_abs_diff_vs_rank0": param_diff, "param_elements_not_bit_identical": param_bits,
            "grad_allreduce_vs_manual_sum_rel": gdiff, "grad_allreduce_vs_manual_sum_rel_l2": gdiff_l2,
            "grad_allreduce_vs_manual_sum_rel_worst_bucket": gdiff_bucket,
            "per_rank_grad_spread_rel": spread, "buckets": len(engine.buckets), "arena_mb": n * 4 / 2 ** 20,
            "allreduce_overlapped_with_backward": bool(engine.overlap),
            "buckets_flushed_early": [k for k, c in enumerate(engine._ready_counts or []) if c > 0]}


def time_iw(cx, batch, K, dtype, steps, warmup, graph=True, full_forward=False, sampler=None, dump=None):
    torch = cx.torch
    import lvae_b200
    from lvae_b200.engine import IWEvaluator, shard_samples
    from lvae_b200.configs import baseline_config
    cfg = baseline_config("mnist12")
    torch.manual_seed(42)
    lvae_b200.manual_seed(1234)            # the same seed on every rank: the evaluator offsets each rank's samples
    model = lvae_b200.LadderVAE(**cfg.kwargs()).cuda()
    if dtype == "bf16":
        model.set_compute_dtype(torch.bfloat16)
    x_host = synthetic_batch(cfg, batch, 0).pin_memory()        # every rank evaluates the SAME image batch
    ev = IWEvaluator(model, batch, use_graph=graph, reuse_bottomup=not full_forward)
    x_dev = x_host.cuda()
    k_warm = max(8, cx.world)
    for _ in range(warmup):
        ev.bound(x_dev, k_warm)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cx.barrier()
    if sampler is not None:
        sampler.start()
    e0.record()
    for _ in range(steps):
        res = ev.bound(x_dev, K)
    e1.record()
    cx.barrier()
    clocks = sampler.stop() if sampler is not None else None
    ms = cx.max_over_ranks(e0.elapsed_time(e1)) / steps
    if dump and cx.rank == 0:
        dump_outputs(dump, {"iw_bound": res.double().cpu().numpy()})
    value = batch / (ms * 1e-3)                                  # images whose K-sample bound completes per second
    cx.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        res = ev.bound(x_host, K)
        res_host = res.cpu()
    torch.cuda.synchronize()
    e2e_ms = cx.max_over_ranks((time.perf_counter() - t0) * 1e3) / steps
    _, k_local = shard_samples(K, cx.rank, cx.world)
    unit = "images/s with a %d-sample bound" % K
    fwd_gflop = CONV_GFLOP["mnist12"][0]
    out = {"metric": "IW-%d evals/s (MNIST 12-layer LVAE)" % K, "value": value, "unit": unit, "n_gpus": cx.world, "steps": steps,
           "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "dtype": dtype,
           "config": iw_config(K, cx.world, batch, full_forward),
           "sample_forwards_per_s": value * K,
           "samples_per_rank": k_local,
           "bound_mean_nats": float(res_host.mean()),
           "e2e": {"value": batch / (e2e_ms * 1e-3), "unit": unit, "h2d_bytes_per_step": x_host.numel() * 4,
                   "d2h_bytes_per_step": res_host.numel() * 4},
           "gpu_launches": (ev.launches_per_sample * k_local + ev.launches_bottomup) * steps,
           "launches_per_sample": ev.launches_per_sample,
           # one sample pass = the top-down half of the forward convolutions (the bottom-up pass runs once per batch)
           "conv_tflops_per_gpu_upper": value * K / cx.world * fwd_gflop / 1e3,
           "clocks": clocks}
    del ev, model
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="train", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the BASELINE config's)")
    ap.add_argument("--iw-samples", type=int, default=1000)
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "f32"],
                    help="bf16: bf16 activations, tcgen05 convs, fp32 accumulation (default); f32: exact fp32 CUDA-core path")
    ap.add_argument("--iw-full-forward", action="store_true",
                    help="IW: recompute the bottom-up pass for every sample like the reference's loop (default: once per batch)")
    ap.add_argument("--no-side-stream", action="store_true", help="keep weight-gradient kernels on the main stream")
    ap.add_argument("--side-streams", type=int, default=3, help="number of side streams the weight-gradient kernels rotate over")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-hbm-rooflines", action="store_true", help="skip the stochastic / likelihood kernel microbenchmarks")
    ap.add_argument("--no-extras", action="store_true",
                    help="train workload: skip the iw / configs / value_f32 / dp_check sub-records (A/B timing runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy into a new or empty DIR (float64; arrays of more than %d "
                         "entries as a fixed seeded sample); the inputs depend on the arguments only" % DUMP_SAMPLE)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    if args.dump_outputs and os.path.isdir(args.dump_outputs) and os.listdir(args.dump_outputs):
        ap.error("--dump-outputs %s is not empty: files of an earlier dump would sit next to this one's" % args.dump_outputs)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    import lvae_b200  # noqa: F401

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cx = Ctx(torch, dist, rank, world, local)
    pk = peaks()
    cfg_name, batch = CONFIGS[args.workload]
    batch = args.batch or batch
    sampler = ClockSampler(local)
    graph = not args.no_graph
    side = 0 if args.no_side_stream else args.side_streams

    if args.workload == "iw":
        line = time_iw(cx, batch, args.iw_samples, args.dtype, args.steps, args.warmup, graph, args.iw_full_forward, sampler,
                       args.dump_outputs)
        line.update({"vs_baseline": None, "data": "synthetic"})
        if rank == 0 and world == 1 and not args.no_hbm_rooflines:
            line["roofline_hbm"] = hbm_rooflines("iw")
        if rank == 0 and not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = {k: v for k, v in cpu_baseline_iw(32, 3).items() if k != "s_per_forward"}
        finish(cx, line)
        return

    main_res = time_train(cx, cfg_name, batch, args.dtype, args.steps, args.warmup, graph, side, True, sampler,
                          shares=not args.no_extras, dp_check=not args.no_extras, dump=args.dump_outputs)
    value = main_res["value"]
    gflop = CONV_GFLOP[cfg_name][1]
    line = {"metric": "train images/s (%s LVAE)" % METRIC_NAME.get(cfg_name, cfg_name),
            "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": main_res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.dtype, "data": "synthetic",
            "config": train_config(cfg_name, batch, world, graph),
            "e2e": main_res["e2e"],
            "gpu_launches": main_res["launches_per_step"] * args.steps,
            "launches_per_step": main_res["launches_per_step"],
            "clocks": main_res["clocks"],
            "peak_mem_gb": main_res["peak_mem_gb"], "loss": main_res["loss"]}
    if "dp_check" in main_res:
        line["dp_check"] = main_res["dp_check"]
    # whole step against the SUSTAINED tensor peak (the step is a long back-to-back run), per GPU
    step_tf = value / world * gflop / 1e3
    line["roofline_step"] = {"bound": "tensor", "achieved": step_tf, "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                             "frac": step_tf / pk["tf_sustained"],
                             "what": "algorithmic conv FLOPs of the whole step (%.3f GFLOP / image, SURVEY.md 8) / step time, "
                                     "against the %s sustained bf16 peak" % (gflop, pk["src"])}
    if rank == 0 and "kernel_shares" in main_res:
        ks = main_res["kernel_shares"]
        line["kernel_shares"] = ks
        # in-step rates of the contraction kernels: forward + dgrad FLOPs (2/3 of the step) over the summed conv_tc time,
        # wgrad FLOPs (1/3) over the summed wgrad time -- CUPTI durations of one replayed step, kernels overlap across streams
        tot = batch * gflop * 1e9
        ins = {}
        t_conv = sum(v["us"] for k, v in ks.items() if isinstance(v, dict) and k.startswith(("conv_tc", "conv_gate_tc", "gate_dgrad_tc")))
        t_wg = sum(v["us"] for k, v in ks.items() if isinstance(v, dict) and k.startswith("wgrad_tc"))
        if t_conv > 0:
            a = tot * 2 / 3 / (t_conv * 1e-6) / 1e12
            ins["conv_tc_fwd_dgrad"] = {"achieved": a, "peak": pk["tf_sustained"], "unit": "TFLOP/s", "frac": a / pk["tf_sustained"], "us_in_step": t_conv}
        if t_wg > 0:
            a = tot / 3 / (t_wg * 1e-6) / 1e12
            ins["wgrad_tc"] = {"achieved": a, "peak": pk["tf_sustained"], "unit": "TFLOP/s", "frac": a / pk["tf_sustained"], "us_in_step": t_wg}
        line["roofline_in_step"] = ins
    if rank == 0:
        line["roofline"] = conv_roofline(torch, pk, args.dtype)
        if world == 1 and not args.no_hbm_rooflines:
            line["roofline_hbm"] = hbm_rooflines(args.workload)
    if not args.no_extras and args.workload == "train":
        # ---- the exact-fp32 mode of the same step (the mode the 1e-4 / 1e-3 parity bounds are stated for) ----
        if args.dtype == "bf16":
            r = time_train(cx, cfg_name, batch, "f32", 4, 3, graph, side, False)
            line["value_f32"] = {k: r[k] for k in ("value", "unit", "ms_per_step", "steps", "warmup", "dtype", "launches_per_step")}
            line["value_f32"]["what"] = "same step, exact fp32 CUDA-core convolutions (parity mode)"
        # ---- the other BASELINE.json training configs, a short timing each ----
        cfgs = {}
        for name, key in (("mnist3", "mnist3_b64"), ("mnist12", "mnist12_b128"), ("celeba20", "celeba20_b64")):
            b = CONFIGS[name][1]
            r = time_train(cx, name, b, "bf16", 8, 3, graph, side, True)
            keep = ("value", "unit", "ms_per_step", "steps", "warmup", "dtype", "per_gpu_batch", "launches_per_step", "peak_mem_gb",
                    "e2e", "conv_tflops_per_gpu")
            cfgs[key] = {k: r[k] for k in keep}
            cfgs[key]["n_gpus"] = world
            cfgs[key]["frac_of_bf16_sustained"] = r["conv_tflops_per_gpu"] / pk["tf_sustained"]
        line["configs"] = cfgs
        # ---- the second half of the metric: IW-1000 on MNIST-12, samples sharded over the ranks ----
        iw = time_iw(cx, CONFIGS["iw"][1], args.iw_samples, "bf16", 1, 3, graph, False)
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            iw["cpu_baseline"] = {k: v for k, v in cpu_baseline_iw(32, 3).items() if k != "s_per_forward"}
        if rank == 0 and world == 1 and not args.no_hbm_rooflines:
            iw["roofline_hbm"] = hbm_rooflines("iw")
        line["iw"] = iw
    if rank == 0 and not args.no_cpu_baseline and world == 1:          # the CPU baseline is a single-GPU-run item (rank 0, N = 1 only)
        cb = cpu_baseline_train(cfg_name, CPU_BATCH, 5)          # ~10 s of CPU work on the box's host cores
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
    finish(cx, line)


def finish(cx, line):
    """The ONE JSON line goes out last, after the process group is gone (NCCL's own INFO lines, if the driver asked for
    them, are then already written)."""
    if cx.world > 1:
        cx.dist.barrier()
        cx.dist.destroy_process_group()
    sys.stderr.flush()
    if cx.rank == 0:
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
