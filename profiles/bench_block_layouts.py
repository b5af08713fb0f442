"""Residual-block layouts on the block node or op by op (ops.set_whole_block) on the B200.

    python profiles/bench_block_layouts.py [--out profiles/bench_block_layouts_r03.txt] [--steps 20] [--rounds 3]

Training: CIFAR-15 kwargs at batch 256 in bf16 with ungated blocks, with 'bacdbac' + dropout None (gated), and with both.
For each variant one TrainEngine (CUDA-graph replay, side-stream weight gradients) per setting of the node, built in the same
process; the two are timed alternately, `rounds` times, `steps` replays each after warm-up, with CUDA events around the
replays.  Also launches per step and the peak memory the engine adds (torch allocator peak over its construction, warm-up and
capture).  IW: MNIST-12 kwargs with ungated blocks, batch 1000, K = 32, graph-replayed evaluator, node on and off alternated."""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def _model(cfg, dtype=torch.bfloat16):
    import lvae_b200
    lvae_b200.manual_seed(0)
    model = lvae_b200.LadderVAE(**cfg.kwargs()).cuda()
    model.set_compute_dtype(dtype)
    return model


def _timed(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def train_variant(lines, name, cfg, steps, rounds, B=256):
    from lvae_b200 import ops
    from lvae_b200.engine import TrainEngine
    x = torch.rand(B, cfg.color_ch, *cfg.img_shape, device="cuda")
    engines = {}
    for node in (True, False):
        ops.set_whole_block(node)
        try:
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            eng = TrainEngine(_model(cfg), B, use_graph=True, wgrad_side_stream=True)
            for _ in range(3):
                eng.step(x)
            torch.cuda.synchronize()
            engines[node] = (eng, (torch.cuda.max_memory_allocated() - base) / 2 ** 30)
        finally:
            ops.set_whole_block(True)
    times = {True: [], False: []}
    for _ in range(rounds):
        for node in (True, False):
            eng = engines[node][0]
            times[node].append(_timed(lambda: eng.step(x), steps))
    for node in (True, False):
        t = times[node]
        lines.append("%-34s node %-3s step %.3f ms (rounds: %s)  launches/step %d  peak +%.2f GiB" % (
            name, "on" if node else "off", sorted(t)[len(t) // 2], " ".join("%.3f" % v for v in t),
            engines[node][0].launches_per_step, engines[node][1]))
    del engines
    torch.cuda.empty_cache()


def iw_bench(lines, rounds, B=1000, K=32):
    import lvae_b200
    from lvae_b200 import ops
    from lvae_b200.engine import IWEvaluator
    from oracle import lvae_oracle as O
    cfg = O.baseline_config("mnist12")
    cfg.gated = False
    x = (torch.rand(B, 1, 28, 28, device="cuda") < 0.15).float()
    evs = {}
    for node in (True, False):
        ops.set_whole_block(node)
        try:
            model = _model(cfg).eval()
            ev = IWEvaluator(model, B, use_graph=True)
            lvae_b200.manual_seed(1)
            evs[node] = (ev, float(ev.bound(x, K).mean()))
        finally:
            ops.set_whole_block(True)
    times = {True: [], False: []}
    for _ in range(rounds):
        for node in (True, False):
            ev = evs[node][0]
            times[node].append(_timed(lambda: ev.bound(x, K), 1))
    for node in (True, False):
        t = sorted(times[node])
        lines.append("IW MNIST-12 ungated B=%d K=%d node %-3s %.2f ms / batch = %.1f images/s (rounds: %s)  bound %.4f" % (
            B, K, "on" if node else "off", t[len(t) // 2], B / (t[len(t) // 2] * 1e-3),
            " ".join("%.2f" % v for v in times[node]), evs[node][1]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_block_layouts_r03.txt"))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_block_layouts: needs the GPU")
    import lvae_b200  # noqa: F401  (loads the library)
    from oracle import lvae_oracle as O
    lines = ["GPU: " + gpu_info()]
    for name, gated, bt, p in (("CIFAR-15 ungated", False, "bacdbacd", 0.2), ("CIFAR-15 bacdbac p=None", True, "bacdbac", None),
                               ("CIFAR-15 ungated bacdbac p=None", False, "bacdbac", None)):
        cfg = O.baseline_config("cifar15")
        cfg.gated, cfg.res_block_type, cfg.dropout = gated, bt, p
        train_variant(lines, name, cfg, a.steps, a.rounds)
        print(lines[-2] + "\n" + lines[-1], flush=True)
    iw_bench(lines, a.rounds)
    text = "\n".join(lines) + "\n"
    print(text, end="")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        fh.write(text)


if __name__ == "__main__":
    main()
