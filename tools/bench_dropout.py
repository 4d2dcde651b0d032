"""Cost of training at the reference's dropout (DESIGN.md section 3.16) on one GPU, everything in one process.

  * the graphed Encoder-Cross-Fusion training step of tools/bench_deterministic.py (4 frames, AdamW): bf16 at p = 0.1
    with torch's nn.Dropout between the kernels (PACKAGE_DROPOUT = False) and on the package path, alternating, and the
    p = 0.0 step as the floor; one fp32 pair in fp32 train-GEMM mode "tf32x3".  Peak memory is
    torch.cuda.max_memory_allocated over one eager step of each configuration;
  * the dropout sites alone, forward + backward at 88 892 rows (4 frames of the COCO pyramid), bf16: linear1 of the
    encoder's feed-forward block (1024 <- 256, ReLU) with the dropout in the GEMM epilogue, as the ReLU GEMM + the
    in-place dropout kernel, and with torch's dropout; add-LayerNorm (256) with the dropout inside the kernel and with
    torch's dropout before it.

    python tools/bench_dropout.py [--rounds 5] [--step-iters 5] [--site-iters 20]

CUDA events, medians over rounds; the card's name and power limit are printed first."""
import argparse
import copy
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch                                                                  # noqa: E402
from torch import nn                                                          # noqa: E402

import bench                                                                  # noqa: E402
from tools.bench_deterministic import card, timed                             # noqa: E402

DEV = torch.device("cuda:0")
ROWS = 88_892


def _lef():
    from dfvod_b200.ops.functions import layer_epilogue_func
    return layer_epilogue_func


def alternate(label, fns, iters, rounds):
    """fns: {name: (setup, fn)}; setup() selects the route before each timing window."""
    times = {k: [] for k in fns}
    for setup, fn in fns.values():
        setup()
        fn()
    for _ in range(rounds):
        for k, (setup, fn) in fns.items():
            setup()
            times[k].append(timed(fn, iters))
    med = {k: statistics.median(v) for k, v in times.items()}
    print(f"{label}: " + "; ".join(f"{k} {med[k]:.3f} ms (spread {min(times[k]):.3f}-{max(times[k]):.3f})" for k in fns),
          flush=True)
    return med


def sites(iters, rounds):
    lef = _lef()
    torch.manual_seed(0)
    bf = torch.bfloat16
    lin = nn.Linear(256, 1024).to(DEV, bf)
    norm = nn.LayerNorm(256).to(DEV, bf)
    drop = nn.Dropout(0.1).train()
    x = torch.randn(ROWS, 256, device=DEV, dtype=bf).requires_grad_(True)
    res = torch.randn(ROWS, 256, device=DEV, dtype=bf).requires_grad_(True)
    g1 = torch.randn(ROWS, 1024, device=DEV, dtype=bf)
    g2 = torch.randn(ROWS, 256, device=DEV, dtype=bf)

    def route(package, fused=True):
        def setup():
            lef.PACKAGE_DROPOUT = package
            lef._relu_dropout_epilogue_wins = lambda n, k: fused
        return setup

    def linear_site():
        torch.autograd.backward(lef.linear_relu(lin, x, drop), g1)

    def norm_site():
        torch.autograd.backward(lef.add_layer_norm(norm, x, res, None, None, dropout=drop), g2)

    keep = lef._relu_dropout_epilogue_wins
    alternate(f"linear1 1024 <- 256 + ReLU + dropout 0.1, {ROWS} rows, bf16, forward + backward",
              {"epilogue": (route(True, True), linear_site), "GEMM + dropout kernel": (route(True, False), linear_site),
               "torch dropout": (route(False), linear_site)}, iters, rounds)
    alternate(f"add-LayerNorm 256 + dropout 0.1, {ROWS} rows, bf16, forward + backward",
              {"package": (route(True), norm_site), "torch dropout": (route(False), norm_site)}, iters, rounds)
    lef._relu_dropout_epilogue_wins = keep
    lef.PACKAGE_DROPOUT = True


def train_steps(step_iters, rounds, dtype, configs):
    """configs: {name: (p, package)}."""
    from dfvod_b200 import data_parallel
    from dfvod_b200.deformable_transformer import DeformableTransformer
    lef = _lef()
    torch.manual_seed(4)
    srcs, masks, poss = bench._pyramid(torch, DEV, bench.COCO_SHAPES, 4, dtype, 40)
    dsrcs, dmasks, dposs = bench._pyramid(torch, DEV, bench.COCO_SHAPES, 4, dtype, 140)
    query = torch.randn(300, 512, generator=torch.Generator().manual_seed(7)).to(DEV, dtype)
    steps, peak, losses = {}, {}, {}
    for name, (p, package) in configs.items():
        torch.manual_seed(4)
        model = DeformableTransformer(num_feature_levels=4, return_intermediate_dec=True, use_depth=True, dropout=p,
                                      depth_type="DepthDeform_encoder_cf_dformer").to(DEV, dtype).train()
        opt = torch.optim.AdamW(model.parameters(), lr=1e-5, fused=True)
        loss_fn = lambda m=model: m(srcs, masks, poss, dsrcs, dmasks, dposs, query)[0].float().square().mean()
        lef.PACKAGE_DROPOUT = package           # the route is fixed when the graph is captured
        opt.zero_grad(set_to_none=True)
        loss_fn().backward()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(DEV)
        base = torch.cuda.memory_allocated(DEV)
        opt.zero_grad(set_to_none=True)
        loss_fn().backward()
        torch.cuda.synchronize()
        peak[name] = (torch.cuda.max_memory_allocated(DEV) - base) / 2 ** 30
        steps[name] = data_parallel.GraphedTrainStep(model, opt, loss_fn)
        losses[name] = [float(steps[name]().detach()) for _ in range(2)]
        lef.PACKAGE_DROPOUT = True
    times = {k: [] for k in steps}
    for _ in range(rounds):
        for k, s in steps.items():
            times[k].append(timed(s, step_iters))
    med = {k: statistics.median(v) for k, v in times.items()}
    dt = str(dtype)[6:]
    for k in steps:
        print(f"graphed train step (Encoder-Cross-Fusion, 4 frames, {dt}, AdamW) {k:<26} {med[k]:8.3f} ms  (spread "
              f"{min(times[k]):.3f}-{max(times[k]):.3f}); eager-step peak above the model {peak[k]:6.2f} GiB; "
              f"losses {', '.join(f'{v:.7g}' for v in losses[k])}", flush=True)
    return med, peak


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--step-iters", type=int, default=5)
    ap.add_argument("--site-iters", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_dropout.py measures on a CUDA device; none is visible")
    print(card(), flush=True)
    sites(args.site_iters, args.rounds)
    train_steps(args.step_iters, args.rounds, torch.bfloat16,
                {"p=0.1 torch dropout": (0.1, False), "p=0.1 package": (0.1, True), "p=0.0": (0.0, True)})
    prev = _lef().set_fp32_train_gemm_mode("tf32x3")
    train_steps(args.step_iters, args.rounds, torch.float32,
                {"p=0.1 torch dropout tf32x3": (0.1, False), "p=0.1 package tf32x3": (0.1, True)})
    _lef().set_fp32_train_gemm_mode(prev)


if __name__ == "__main__":
    main()
