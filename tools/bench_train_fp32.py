"""fp32 training linears on one B200: the IEEE SGEMM path (g @ W, g^T @ x, column_sum; TF32 off) against the three-term
TF32 kernels (linear_tf32x3 on the split of W^T for dx, linear_tf32x3_wgrad for dW and db in one pass over g), per shape
and in the whole graphed Encoder-Cross-Fusion training step of bench.py in fp32, set_fp32_train_gemm_mode("library")
against ("tf32x3").

    python tools/bench_train_fp32.py [--iters 30] [--rounds 5] [--step-iters 5] [--profile] [--errors-only]

Both sides alternate in one process, timed with CUDA events; medians over rounds.  Errors are normalised max errors
against the fp64 product of the same fp32 operands; plain library TF32 (one TF32 GEMM) is printed for context only.
--errors-only prints the weight-gradient errors and nothing else (to compare builds, e.g. another accumulator chunk
length through MSDA_B200_LIB).  --profile adds one eager fp32 training step in mode "tf32x3" under torch.profiler and
lists the library GEMM calls that have the encoder's row count."""
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
ROWS = [2400, 88892, 177784]                                                  # decoder-sized; 4 and 8 frames of COCO


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
    return float((a.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-300))


class tf32_matmul:
    def __init__(self, on):
        self.on = on

    def __enter__(self):
        self.prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = self.on

    def __exit__(self, *exc):
        torch.backends.cuda.matmul.allow_tf32 = self.prev


def operands(rows, n, k):
    torch.manual_seed(rows + n + k)
    g = torch.randn(rows, n, device=DEV) / 4
    x = torch.randn(rows, k, device=DEV) * 2
    w = torch.randn(n, k, device=DEV) / 16
    b = torch.randn(n, device=DEV)
    return g, x, w, b


def errors_only():
    print("weight-gradient error against fp64 (normalised max): dW kernel | dW SGEMM | db kernel | db sum")
    for rows in ROWS:
        for n, k in SHAPES:
            g, x, _, _ = operands(rows, n, k)
            dw, db = L.linear_tf32x3_wgrad(g, x)
            with tf32_matmul(False):
                sg = g.t() @ x
            rw, rb = g.double().t() @ x.double(), g.double().sum(0)
            print(f"{rows:>7} {n:>5} {k:>5} | {nerr(dw, rw):.2e} | {nerr(sg, rw):.2e} | {nerr(db, rb):.2e} | "
                  f"{nerr(g.sum(0), rb):.2e}", flush=True)


def per_shape(iters, rounds):
    print(f"{'rows':>7} {'out':>5} {'in':>5} | backward {'SGEMM us':>9} {'kernels us':>10} {'speedup':>7} | "
          f"forward {'SGEMM us':>9} {'kernel us':>9} {'speedup':>7} | error vs fp64 dx / dW / db: SGEMM | kernels | "
          f"(TF32 library)")
    for rows in ROWS:
        for n, k in SHAPES:
            g, x, w, b = operands(rows, n, k)
            w_hi, w_lo = L._tf32_weight_split(w)

            def lib_bwd():
                with tf32_matmul(False):
                    return g @ w, g.t() @ x, L.column_sum(g)

            def own_bwd():                               # what the route does in a backward, W^T split included
                return (L._linear_tf32x3_kernel(g, w_hi.t().contiguous(), w_lo.t().contiguous(), None),) + \
                    L.linear_tf32x3_wgrad(g, x)

            def lib_fwd():
                with tf32_matmul(False):
                    return torch.addmm(b, x, w.t())

            own_fwd = lambda: L._linear_tf32x3_kernel(x, w_hi, w_lo, b)
            refs = (g.double() @ w.double(), g.double().t() @ x.double(), g.double().sum(0))
            with tf32_matmul(True):
                tf32 = (g @ w, g.t() @ x)
            errs = [" / ".join(f"{nerr(p, r):.1e}" for p, r in zip(side, refs)) for side in (lib_bwd(), own_bwd())]
            errs.append(" / ".join(f"{nerr(p, r):.1e}" for p, r in zip(tf32, refs)))
            fns = (lib_bwd, own_bwd, lib_fwd, own_fwd)
            for fn in fns:
                timed(fn, 3)
            t = [[] for _ in fns]
            for _ in range(rounds):
                for i, fn in enumerate(fns):
                    t[i].append(timed(fn, iters))
            m = [statistics.median(v) * 1e3 for v in t]
            print(f"{rows:>7} {n:>5} {k:>5} | backward {m[0]:>9.1f} {m[1]:>10.1f} {m[0] / m[1]:>7.3f} | "
                  f"forward {m[2]:>9.1f} {m[3]:>9.1f} {m[2] / m[3]:>7.3f} | {errs[0]} | {errs[1]} | ({errs[2]})",
                  flush=True)
            del g, x, w, b, w_hi, w_lo


def train_model():
    from dfvod_b200.deformable_transformer import DeformableTransformer
    torch.manual_seed(4)
    model = DeformableTransformer(num_feature_levels=4, return_intermediate_dec=True, use_depth=True, dropout=0.0,
                                  depth_type="DepthDeform_encoder_cf_dformer").to(DEV)
    f32 = torch.float32
    srcs, masks, poss = bench._pyramid(torch, DEV, bench.COCO_SHAPES, 4, f32, 40)
    dsrcs, dmasks, dposs = bench._pyramid(torch, DEV, bench.COCO_SHAPES, 4, f32, 140)
    query = torch.randn(300, 512, generator=torch.Generator().manual_seed(7)).to(DEV, f32)
    return model, (srcs, masks, poss, dsrcs, dmasks, dposs, query)


def whole_step(step_iters, rounds):
    from dfvod_b200 import data_parallel
    base, inputs = train_model()
    steps = {}
    with tf32_matmul(False):
        for mode in ("library", "tf32x3"):
            model = copy.deepcopy(base)
            opt = torch.optim.AdamW(model.parameters(), lr=1e-5, fused=True)
            prev = L.set_fp32_train_gemm_mode(mode)       # the route is fixed when the graph is captured
            loss_fn = lambda m=model: m(*inputs)[0].square().mean()
            for _ in range(2):                           # eager warm-up (shape caches read spatial_shapes back once)
                opt.zero_grad(set_to_none=True)
                loss_fn().backward()
            steps[mode] = data_parallel.GraphedTrainStep(model, opt, loss_fn)
            L.set_fp32_train_gemm_mode(prev)
        losses = {k: [float(s().detach()) for _ in range(3)] for k, s in steps.items()}
        times = {k: [] for k in steps}
        for _ in range(rounds):
            for k, s in steps.items():
                times[k].append(timed(s, step_iters))
    med = {k: statistics.median(v) for k, v in times.items()}
    print(f"graphed train_step (DepthDeform_encoder_cf_dformer, 4 frames, fp32, AdamW), threshold "
          f"{L.FP32_TRAIN_KERNEL_MIN_ROWS} rows: library {med['library']:.3f} ms, tf32x3 {med['tf32x3']:.3f} ms per step "
          f"(spread library {min(times['library']):.3f}-{max(times['library']):.3f}, "
          f"tf32x3 {min(times['tf32x3']):.3f}-{max(times['tf32x3']):.3f}; {rounds} rounds of {step_iters} steps)",
          flush=True)
    print(f"first losses library {', '.join(f'{v:.7g}' for v in losses['library'])}; "
          f"tf32x3 {', '.join(f'{v:.7g}' for v in losses['tf32x3'])}", flush=True)


def profile_step():
    from torch.profiler import ProfilerActivity, profile
    model, inputs = train_model()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-5, fused=True)

    def step():
        opt.zero_grad(set_to_none=True)
        model(*inputs)[0].square().mean().backward()
        opt.step()

    prev = L.set_fp32_train_gemm_mode("tf32x3")
    with tf32_matmul(False):
        for _ in range(2):
            step()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA], record_shapes=True) as prof:
            step()
            torch.cuda.synchronize()
    L.set_fp32_train_gemm_mode(prev)
    big = 88892
    gemms = {}
    for e in prof.events():
        if e.name in ("aten::mm", "aten::addmm", "aten::_addmm_activation", "aten::matmul") and e.input_shapes:
            if any(big in s for s in e.input_shapes if s):
                gemms[(e.name, str(e.input_shapes))] = gemms.get((e.name, str(e.input_shapes)), 0) + 1
    print(f"library GEMM calls with {big} rows in one eager fp32 training step, mode tf32x3 "
          f"(threshold {L.FP32_TRAIN_KERNEL_MIN_ROWS}): {sum(gemms.values())}")
    for (name, shapes), c in sorted(gemms.items()):
        print(f"  {c:>3} x {name} {shapes}")
    names = {}
    for e in prof.key_averages():
        if "linear_tf32x3" in e.key or "gemm" in e.key.lower() or "nvjet" in e.key.lower():
            names[e.key] = (e.count, e.device_time_total / 1e3)
    print("GEMM-like kernels of the step (launches, device ms):")
    for k, (c, ms) in sorted(names.items(), key=lambda kv: -kv[1][1]):
        print(f"  {c:>4} {ms:>8.2f}  {k[:100]}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--step-iters", type=int, default=5)
    ap.add_argument("--skip-shapes", action="store_true")
    ap.add_argument("--skip-step", action="store_true")
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--errors-only", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_train_fp32.py measures on a CUDA device; none is visible")
    print(card(), flush=True)
    if args.errors_only:
        errors_only()
        return
    if not args.skip_shapes:
        per_shape(args.iters, args.rounds)
    if not args.skip_step:
        whole_step(args.step_iters, args.rounds)
    if args.profile:
        profile_step()


if __name__ == "__main__":
    main()
