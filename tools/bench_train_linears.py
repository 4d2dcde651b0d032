"""bf16 training linears on one B200: the library backward (g @ W, g^T @ x, column_sum) against the package's kernels
(linear_bf16 on W^T for dx, linear_bf16_wgrad for dW and db in one pass over g), per shape and in the whole graphed
Encoder-Cross-Fusion training step of bench.py (train_step).

    python tools/bench_train_linears.py [--iters 50] [--rounds 5] [--step-iters 10] [--profile]

Both sides alternate in one process, timed with CUDA events; medians over rounds.  --profile adds one eager training step
under torch.profiler with shapes recorded and lists the library GEMM calls that have the encoder's row count."""
import argparse
import copy
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch                                                                  # noqa: E402

import bench                                                                  # noqa: E402
from dfvod_b200.ops.functions import layer_epilogue_func as L                 # noqa: E402

DEV = torch.device("cuda:0")
SHAPES = [(256, 256), (384, 256), (1024, 256), (256, 1024)]                   # (out, in)
ROWS = [88892, 177784]                                                        # 4 and 8 frames of the COCO pyramid


def card():
    name = torch.cuda.get_device_name(DEV)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "power limit unknown"
    return f"{name}, {q}"


def timed(fn, iters):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / iters


def nerr(a, ref):
    return float((a.double() - ref.double()).abs().max() / ref.double().abs().max().clamp_min(1e-300))


def per_shape(iters, rounds):
    print(f"{'rows':>7} {'out':>5} {'in':>5} | {'library us':>10} {'GB/s':>6} | {'kernels us':>10} {'GB/s':>6} | "
          f"{'speedup':>7} | agreement dx / dW / db (normalised max)")
    for rows in ROWS:
        for n, k in SHAPES:
            torch.manual_seed(rows + n + k)
            g = torch.randn(rows, n, device=DEV).bfloat16()
            x = torch.randn(rows, k, device=DEV).bfloat16()
            w = (torch.randn(n, k, device=DEV) / 16).bfloat16()
            lib = lambda: (g @ w, g.t() @ x, L.column_sum(g))
            own = lambda: (L.linear_bf16(g, w.t().contiguous(), None),) + L.linear_bf16_wgrad(g, x)
            a, b = lib(), own()
            agree = " / ".join(f"{nerr(p, q):.1e}" for p, q in zip(b, a))
            for fn in (lib, own):
                timed(fn, 5)
            t_lib, t_own = [], []
            for _ in range(rounds):
                t_lib.append(timed(lib, iters))
                t_own.append(timed(own, iters))
            ml, mo = statistics.median(t_lib) * 1e3, statistics.median(t_own) * 1e3
            # bytes the algorithm needs: read g, x, W once; write dx, dW, db once
            need = 2 * (rows * n + rows * k + n * k + rows * k + n * k + n)
            print(f"{rows:>7} {n:>5} {k:>5} | {ml:>10.1f} {need / ml / 1e3:>6.0f} | {mo:>10.1f} {need / mo / 1e3:>6.0f} | "
                  f"{ml / mo:>7.3f} | {agree}", flush=True)


def train_model():
    from dfvod_b200.deformable_transformer import DeformableTransformer
    torch.manual_seed(4)
    model = DeformableTransformer(num_feature_levels=4, return_intermediate_dec=True, use_depth=True, dropout=0.0,
                                  depth_type="DepthDeform_encoder_cf_dformer").to(DEV).bfloat16()
    bf = torch.bfloat16
    srcs, masks, poss = bench._pyramid(torch, DEV, bench.COCO_SHAPES, 4, bf, 40)
    dsrcs, dmasks, dposs = bench._pyramid(torch, DEV, bench.COCO_SHAPES, 4, bf, 140)
    query = torch.randn(300, 512, generator=torch.Generator().manual_seed(7)).to(DEV, bf)
    return model, (srcs, masks, poss, dsrcs, dmasks, dposs, query)


def whole_step(step_iters, rounds):
    from dfvod_b200 import data_parallel
    default = L.BF16_TRAIN_KERNEL_MIN_ROWS
    base, inputs = train_model()
    steps = {}
    for label, threshold in (("library", None), ("kernels", default)):
        model = copy.deepcopy(base)
        opt = torch.optim.AdamW(model.parameters(), lr=1e-5, fused=True)
        L.BF16_TRAIN_KERNEL_MIN_ROWS = threshold          # the route is fixed when the graph is captured
        loss_fn = lambda m=model: m(*inputs)[0].float().square().mean()
        for _ in range(2):                               # eager warm-up (shape caches read spatial_shapes back once)
            opt.zero_grad(set_to_none=True)
            loss_fn().backward()
        steps[label] = data_parallel.GraphedTrainStep(model, opt, loss_fn)
    L.BF16_TRAIN_KERNEL_MIN_ROWS = default
    losses = {k: float(s().detach()) for k, s in steps.items()}
    times = {k: [] for k in steps}
    for _ in range(rounds):
        for k, s in steps.items():
            times[k].append(timed(s, step_iters))
    med = {k: statistics.median(v) for k, v in times.items()}
    print(f"graphed train_step (DepthDeform_encoder_cf_dformer, 4 frames, bf16, AdamW), threshold {default} rows: "
          f"library {med['library']:.3f} ms, kernels {med['kernels']:.3f} ms per step "
          f"(spread library {min(times['library']):.3f}-{max(times['library']):.3f}, "
          f"kernels {min(times['kernels']):.3f}-{max(times['kernels']):.3f}); "
          f"first losses {losses['library']:.6g} / {losses['kernels']:.6g}", flush=True)


def profile_step():
    from torch.profiler import ProfilerActivity, profile
    model, inputs = train_model()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-5, fused=True)

    def step():
        opt.zero_grad(set_to_none=True)
        model(*inputs)[0].float().square().mean().backward()
        opt.step()

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA], record_shapes=True) as prof:
        step()
        torch.cuda.synchronize()
    big = 88892
    gemms = {}
    for e in prof.events():
        if e.name in ("aten::mm", "aten::addmm", "aten::_addmm_activation", "aten::matmul") and e.input_shapes:
            if any(big in s for s in e.input_shapes if s):
                gemms[(e.name, str(e.input_shapes))] = gemms.get((e.name, str(e.input_shapes)), 0) + 1
    print(f"library GEMM calls with {big} rows in one eager training step "
          f"(threshold {L.BF16_TRAIN_KERNEL_MIN_ROWS}): {sum(gemms.values())}")
    for (name, shapes), c in sorted(gemms.items()):
        print(f"  {c:>3} x {name} {shapes}")
    names = {}
    for e in prof.key_averages():
        if "linear_bf16" in e.key or "gemm" in e.key.lower() or "nvjet" in e.key.lower():
            names[e.key] = e.count
    print("GEMM-like kernels of the step (name: launches):")
    for k, c in sorted(names.items(), key=lambda kv: -kv[1]):
        print(f"  {c:>4}  {k[:110]}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--step-iters", type=int, default=10)
    ap.add_argument("--skip-shapes", action="store_true")
    ap.add_argument("--skip-step", action="store_true")
    ap.add_argument("--profile", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_train_linears.py measures on a CUDA device; none is visible")
    print(card(), flush=True)
    if not args.skip_shapes:
        per_shape(args.iters, args.rounds)
    if not args.skip_step:
        whole_step(args.step_iters, args.rounds)
    if args.profile:
        profile_step()


if __name__ == "__main__":
    main()
