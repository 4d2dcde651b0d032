"""Cost of the deterministic backward (DESIGN.md section 3.15) on one GPU: the default backward (fp32 vector atomics)
against the deterministic one (fixed-point int64 reductions), alternating in one process.

  * the op backward at the COCO encoder shape (batch 8, S = Lq = 22 223, 8 heads of 32, 4 levels x 4 points, encoder
    geometry), plain op (MSDA.ms_deform_attn_backward) and fused op (MSDeformAttnFusedFunction), fp32 and bf16;
  * the graphed Encoder-Cross-Fusion training step of tools/profile_train_step.py (bf16, 4 frames, AdamW), one graph
    captured with torch.use_deterministic_algorithms off and one with it on (warn_only: the decoder's attention is
    torch's own and outside this package's guarantee).

    python tools/bench_deterministic.py [--iters 20] [--rounds 5] [--step-iters 5] [--no-step] [--profile]

--profile adds a torch.profiler table of the kernels of one deterministic fp32 plain backward (pre-pass, accumulation,
finishing kernel) after the timings.

The op timings run with torch.utils.deterministic.fill_uninitialized_memory off, so they time the package's kernels
and not torch's NaN fill of freshly allocated outputs; the training step keeps torch's default.  CUDA events, medians
over rounds, the card's name and power limit printed first."""
import argparse
import copy
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")     # before cuBLAS starts: deterministic library GEMMs
import torch                                                                  # noqa: E402

import bench                                                                  # noqa: E402

DEV = torch.device("cuda:0")


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


def set_mode(det):
    torch.use_deterministic_algorithms(det, warn_only=True)


def compare(label, fn, iters, rounds):
    """fn() runs one backward under the current mode; returns the gradients of the last call of each mode."""
    times = {False: [], True: []}
    last = {}
    for det in (False, True):               # warm-up
        set_mode(det)
        last[det] = fn()
    for _ in range(rounds):
        for det in (False, True):
            set_mode(det)
            times[det].append(timed(fn, iters))
    set_mode(False)
    med = {k: statistics.median(v) for k, v in times.items()}
    diff = float((last[True].double() - last[False].double()).abs().max() / last[False].double().abs().max())
    print(f"{label:<28} default {med[False]:8.3f} ms  deterministic {med[True]:8.3f} ms  ratio {med[True] / med[False]:5.2f}"
          f"  (spread {min(times[False]):.3f}-{max(times[False]):.3f} / {min(times[True]):.3f}-{max(times[True]):.3f};"
          f" grad_value normalised max difference {diff:.2e})", flush=True)


def op_backwards(iters, rounds):
    from dfvod_b200 import MultiScaleDeformableAttention as MSDA
    from dfvod_b200.ops.functions import MSDeformAttnFusedFunction
    n, m, nl, p = 8, bench.M, len(bench.COCO_SHAPES), bench.P
    value, loc, attn, gout = bench.make_inputs(torch, n, 0, "grid")
    lsi, s = bench.level_start(bench.COCO_SHAPES)
    st = torch.as_tensor(bench.COCO_SHAPES, dtype=torch.long, device=DEV)
    ls = torch.as_tensor(lsi, dtype=torch.long, device=DEV)
    loc, attn = loc.to(DEV), attn.to(DEV)
    # fused: the same geometry as raw projection outputs (offsets in pixels, logits), points as reference
    g = torch.Generator().manual_seed(1)
    ref = torch.rand(n, s, nl, 2, generator=g).to(DEV)
    raw = (torch.randn(n, s, 3 * m * nl * p, generator=g) * 2.0).to(DEV)
    for dtype in (torch.float32, torch.bfloat16):
        v, go = value.to(DEV, dtype), gout.to(DEV, dtype)
        compare(f"plain backward {str(dtype)[6:]}",
                lambda: MSDA.ms_deform_attn_backward(v, st, ls, loc, attn, go, 64)[0], iters, rounds)
        vr = v.clone().requires_grad_(True)
        rr = raw.to(dtype).requires_grad_(True)
        rf = ref.clone().requires_grad_(True)
        out = MSDeformAttnFusedFunction.apply(vr, st, ls, rf, rr, p)

        def fused():
            (gv,) = torch.autograd.grad(out, vr, go, retain_graph=True)
            return gv
        compare(f"fused backward {str(dtype)[6:]}", fused, iters, rounds)
        del v, go, vr, rr, rf, out
    torch.cuda.empty_cache()


def profile_plain():
    from torch.profiler import ProfilerActivity, profile
    from dfvod_b200 import MultiScaleDeformableAttention as MSDA
    value, loc, attn, gout = (t.to(DEV) for t in bench.make_inputs(torch, 8, 0, "grid"))
    lsi, _ = bench.level_start(bench.COCO_SHAPES)
    st = torch.as_tensor(bench.COCO_SHAPES, dtype=torch.long, device=DEV)
    ls = torch.as_tensor(lsi, dtype=torch.long, device=DEV)
    set_mode(True)
    for _ in range(2):
        MSDA.ms_deform_attn_backward(value, st, ls, loc, attn, gout, 64)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            MSDA.ms_deform_attn_backward(value, st, ls, loc, attn, gout, 64)
        torch.cuda.synchronize()
    set_mode(False)
    print("deterministic fp32 plain backward, 5 calls:", flush=True)
    print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=10, max_name_column_width=60), flush=True)


def train_step(step_iters, rounds):
    from dfvod_b200 import data_parallel
    from dfvod_b200.deformable_transformer import DeformableTransformer
    torch.manual_seed(4)
    base = DeformableTransformer(num_feature_levels=4, return_intermediate_dec=True, use_depth=True, dropout=0.0,
                                 depth_type="DepthDeform_encoder_cf_dformer").to(DEV).bfloat16()
    bf = torch.bfloat16
    srcs, masks, poss = bench._pyramid(torch, DEV, bench.COCO_SHAPES, 4, bf, 40)
    dsrcs, dmasks, dposs = bench._pyramid(torch, DEV, bench.COCO_SHAPES, 4, bf, 140)
    query = torch.randn(300, 512, generator=torch.Generator().manual_seed(7)).to(DEV, bf)
    steps = {}
    for det in (False, True):
        model = copy.deepcopy(base)
        opt = torch.optim.AdamW(model.parameters(), lr=1e-5, fused=True)
        loss_fn = lambda m=model: m(srcs, masks, poss, dsrcs, dmasks, dposs, query)[0].float().square().mean()
        set_mode(det)                          # the route is fixed when the graph is captured
        for _ in range(2):
            opt.zero_grad(set_to_none=True)
            loss_fn().backward()
        steps[det] = data_parallel.GraphedTrainStep(model, opt, loss_fn)
        set_mode(False)
    losses = {k: [float(s().detach()) for _ in range(3)] for k, s in steps.items()}
    times = {k: [] for k in steps}
    for _ in range(rounds):
        for k, s in steps.items():
            times[k].append(timed(s, step_iters))
    med = {k: statistics.median(v) for k, v in times.items()}
    print(f"graphed train step (Encoder-Cross-Fusion, 4 frames, bf16, AdamW): default {med[False]:.3f} ms, "
          f"deterministic {med[True]:.3f} ms, ratio {med[True] / med[False]:.3f} (spread "
          f"{min(times[False]):.3f}-{max(times[False]):.3f} / {min(times[True]):.3f}-{max(times[True]):.3f}; "
          f"{rounds} rounds of {step_iters} steps)", flush=True)
    print(f"first losses default {', '.join(f'{v:.7g}' for v in losses[False])}; "
          f"deterministic {', '.join(f'{v:.7g}' for v in losses[True])}", flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--step-iters", type=int, default=5)
    ap.add_argument("--no-step", action="store_true", help="time only the op backwards")
    ap.add_argument("--profile", action="store_true", help="kernel table of one deterministic backward")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_deterministic.py measures on a CUDA device; none is visible")
    print(card(), flush=True)
    fill = torch.utils.deterministic.fill_uninitialized_memory
    torch.utils.deterministic.fill_uninitialized_memory = False
    op_backwards(args.iters, args.rounds)
    if args.profile:
        profile_plain()
    torch.utils.deterministic.fill_uninitialized_memory = fill
    if not args.no_step:
        train_step(args.step_iters, args.rounds)


if __name__ == "__main__":
    main()
