"""128-filter tensor-core path on the B200: the 3x3 128 -> 128 convolution (forward and data gradient on streamed weights,
weight gradient over 2 X windows x 2 dY windows) and the CIFAR-15 training step at n_filters = 128.

    python profiles/bench_wide.py [--out profiles/bench_wide_r03.txt] [--steps 5]

Kernel times: CUDA-graph replay of 20 launches rotating over operand sets larger than the 126 MB L2, CUDA events around
the replay; TFLOP/s from the shapes (2 * B * H * W * 9 * 128 * 128 per pass).  Step times: TrainEngine (graph replay,
side-stream weight gradients) in bf16, and the fp32 parity mode (CUDA-core kernels), after warm-up."""
import argparse
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def time_graph(fn, reps=20, iters=5):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for i in range(3):
            fn(i)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(reps):
            fn(i)
    g.replay()
    torch.cuda.synchronize()
    best = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        g.replay()
        b.record()
        b.synchronize()
        best.append(a.elapsed_time(b) / reps)
    best.sort()
    return best[len(best) // 2], best[0], best[-1]


def conv_bench(lines):
    from lvae_b200 import ops
    from lvae_b200.lib.nn import Conv2d
    conv = Conv2d(128, 128, 3, padding=1).cuda()
    sp = conv.spec
    for H in (16, 32):
        B = 256
        nbytes = B * H * H * 128 * 2
        nset = max(2, -(-3 * 126 * 2 ** 20 // (2 * nbytes)))          # x and dY sets together > 3 x L2
        xs = [torch.randn(B, H, H, 128, device="cuda").to(torch.bfloat16) for _ in range(nset)]
        gys = [torch.randn(B, H, H, 128, device="cuda").to(torch.bfloat16) for _ in range(nset)]
        wpf = sp.pack_tc_fwd.get(conv.weight, torch.bfloat16)
        wpb = sp.pack_tc_bwd.get(conv.weight, torch.bfloat16)
        dw = torch.zeros(128, 128, 3, 3, device="cuda")
        db = torch.zeros(128, device="cuda")
        ws = torch.empty(512 * 128, device="cuda")
        st = lambda: torch.cuda.current_stream().cuda_stream
        flops = 2.0 * B * H * H * 9 * 128 * 128
        plan = ops.conv_tc_plan(128, 128, 3, False, H, H, False)

        def fwd(i):
            ops._conv_tc(xs[i % nset], None, wpf, conv.bias, None, None, 128, 3, False, False)

        def dgrad(i):
            ops._conv_tc(gys[i % nset], None, wpb, None, None, None, 128, 3, True, False)

        def wgrad(i):
            for x0, n, c0 in ops.wgrad_tc_windows(128, 3, False, 128):
                ops.call("lvae_conv2d_wgrad_tc_ex", xs[i % nset].data_ptr(), None, gys[i % nset].data_ptr(),
                         dw.data_ptr() + c0 * 128 * 9 * 4, None if x0 else db.data_ptr() + c0 * 4, ws.data_ptr(),
                         B, H, H, n, 3, 0, 0, 128, c0, 128, x0, st())
        for name, fn in (("forward (streamed)" if plan == 2 else "forward", fwd), ("dgrad", dgrad),
                         ("wgrad (2 X x 2 dY windows)", wgrad)):
            med, lo, hi = time_graph(fn)
            lines.append("3x3 128->128 B=%d %dx%d %-28s %8.1f us (min %.1f max %.1f)  %6.0f TFLOP/s" % (
                B, H, H, name, med * 1e3, lo * 1e3, hi * 1e3, flops / (med * 1e-3) / 1e12))
        del xs, gys
        torch.cuda.empty_cache()


def step_bench(lines, steps, dtype):
    import lvae_b200
    from lvae_b200.engine import TrainEngine
    from oracle import lvae_oracle as O
    cfg = O.baseline_config("cifar15")
    cfg.n_filters = 128
    lvae_b200.manual_seed(0)
    model = lvae_b200.LadderVAE(**cfg.kwargs()).cuda()
    if dtype == torch.bfloat16:
        model.set_compute_dtype(torch.bfloat16)
    B = 256
    eng = TrainEngine(model, B, use_graph=dtype == torch.bfloat16, wgrad_side_stream=dtype == torch.bfloat16)
    x = torch.rand(B, 3, 32, 32, device="cuda")
    for _ in range(3):
        eng.step(x)
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(steps):
        out = eng.step(x)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t) / steps
    lines.append("CIFAR-15 n_filters=128 batch %d %-5s step %8.2f ms  (%d steps after 3 warm-up; loss %.4f)" % (
        B, "bf16" if dtype == torch.bfloat16 else "fp32", dt * 1e3, steps, float(out["loss"])))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_wide_r03.txt"))
    ap.add_argument("--steps", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_wide: needs the GPU")
    import lvae_b200  # noqa: F401  (builds / loads the library)
    lines = ["GPU: " + gpu_info()]
    conv_bench(lines)
    step_bench(lines, a.steps, torch.bfloat16)
    step_bench(lines, max(1, a.steps // 2), torch.float32)
    text = "\n".join(lines) + "\n"
    print(text, end="")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        fh.write(text)


if __name__ == "__main__":
    main()
