"""Cost of Deformable DETR's matching and set criterion (DESIGN.md section 3.17) on one GPU, in one process.

  * the matcher alone: final + 5 auxiliary decoder heads (6 decoder layers), Q = 300, 91 classes, B images with T
    boxes each.  Device: dfvod_b200.HungarianMatcher.match_padded (cost on the GPU, one solver launch, nothing read
    back).  Reference: oracle/criterion_oracle.HungarianMatcher per head (cost on the GPU, .cpu(), scipy per image).
    Host clock around each call, ending in a device synchronise;
  * the SURVEY C5 training step (Encoder-Cross-Fusion transformer, bf16, 4 frames, AdamW, COCO pyramid) with
    Deformable DETR's class and box heads and the full criterion (6 decoder heads, 91 classes, 4..30 boxes per frame):
    the graphed step (data_parallel.GraphedTrainStep) with dfvod_b200.SetCriterion on padded targets against the eager
    step with the reference-form criterion (oracle matcher, .item() on the box count).

    python tools/bench_criterion.py [--rounds 5] [--iters 20] [--step-iters 5]

Medians over rounds; the card's name and power limit are printed first."""
import argparse
import copy
import os
import statistics
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch                                                                  # noqa: E402

import bench                                                                  # noqa: E402
from tools.bench_deterministic import card, timed                             # noqa: E402

DEV = torch.device("cuda:0")
NUM_CLASSES = 91
WEIGHTS = {"loss_ce": 2.0, "loss_bbox": 5.0, "loss_giou": 2.0}


def host_timed(fn, iters):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / iters


def make_targets(g, counts):
    return [{"labels": torch.randint(0, NUM_CLASSES, (n,), generator=g).to(DEV),
             "boxes": torch.cat([torch.rand(n, 2, generator=g) * 0.8 + 0.1,
                                 torch.rand(n, 2, generator=g) * 0.3 + 0.02], 1).to(DEV)} for n in counts]


def matcher(iters, rounds):
    import dfvod_b200
    from oracle import criterion_oracle
    mine, ref = dfvod_b200.HungarianMatcher(2, 5, 2), criterion_oracle.HungarianMatcher(2, 5, 2)
    g = torch.Generator().manual_seed(0)
    for b in (4, 8):
        for t in (5, 30, 100):
            heads = [{"pred_logits": (torch.randn(b, 300, NUM_CLASSES, generator=g) * 2 - 3).to(DEV),
                      "pred_boxes": torch.randn(b, 300, 4, generator=g).sigmoid().to(DEV)} for _ in range(6)]
            targets = make_targets(g, [t] * b)
            padded = dfvod_b200.pad_targets(targets, t)
            fns = {"device": lambda: mine.match_padded([(h, padded.labels, padded) for h in heads]),
                   "cpu scipy": lambda: [ref(h, targets) for h in heads]}
            times = {k: [] for k in fns}
            for fn in fns.values():
                fn()
            for _ in range(rounds):
                for k, fn in fns.items():
                    times[k].append(host_timed(fn, iters))
            med = {k: statistics.median(v) for k, v in times.items()}
            print(f"matcher B={b} Q=300 T={t} x 6 heads: device {med['device']:.3f} ms "
                  f"(spread {min(times['device']):.3f}-{max(times['device']):.3f}); .cpu() + scipy "
                  f"{med['cpu scipy']:.3f} ms (spread {min(times['cpu scipy']):.3f}-{max(times['cpu scipy']):.3f})",
                  flush=True)


def weighted(losses):
    base = lambda k: k if k in WEIGHTS else k.rsplit("_", 1)[0]
    return sum(v * WEIGHTS[base(k)] for k, v in losses.items() if base(k) in WEIGHTS)


class Detector(torch.nn.Module):
    """Deformable DETR's heads (class head, 3-layer box MLP, no box refinement) on the C5 transformer."""

    def __init__(self, transformer):
        super().__init__()
        self.transformer = transformer
        self.class_embed = torch.nn.Linear(256, NUM_CLASSES)
        self.bbox_embed = torch.nn.Sequential(torch.nn.Linear(256, 256), torch.nn.ReLU(), torch.nn.Linear(256, 256),
                                              torch.nn.ReLU(), torch.nn.Linear(256, 4))

    def forward(self, srcs, masks, poss, dsrcs, dmasks, dposs, query):
        hs, init_ref, inter_refs, _, _ = self.transformer(srcs, masks, poss, dsrcs, dmasks, dposs, query)
        classes, coords = [], []
        for lvl in range(hs.shape[0]):
            ref = (init_ref if lvl == 0 else inter_refs[lvl - 1]).float().clamp(1e-5, 1 - 1e-5)
            tmp = self.bbox_embed(hs[lvl]).float()
            coords.append(torch.cat([tmp[..., :2] + torch.log(ref / (1 - ref)), tmp[..., 2:]], -1).sigmoid())
            classes.append(self.class_embed(hs[lvl]).float())
        return {"pred_logits": classes[-1], "pred_boxes": coords[-1],
                "aux_outputs": [{"pred_logits": a, "pred_boxes": b} for a, b in zip(classes[:-1], coords[:-1])]}


def train_step(step_iters, rounds):
    import dfvod_b200
    from dfvod_b200 import data_parallel
    from dfvod_b200.deformable_transformer import DeformableTransformer
    from oracle import criterion_oracle
    torch.manual_seed(4)
    bf = torch.bfloat16
    transformer = DeformableTransformer(num_feature_levels=4, return_intermediate_dec=True, use_depth=True, dropout=0.0,
                                        depth_type="DepthDeform_encoder_cf_dformer")
    model = Detector(transformer).to(DEV).bfloat16()
    srcs, masks, poss = bench._pyramid(torch, DEV, bench.COCO_SHAPES, 4, bf, 40)
    dsrcs, dmasks, dposs = bench._pyramid(torch, DEV, bench.COCO_SHAPES, 4, bf, 140)
    query = torch.randn(300, 512, generator=torch.Generator().manual_seed(7)).to(DEV, bf)
    targets = make_targets(torch.Generator().manual_seed(3), [4, 30, 17, 9])
    losses = ["labels", "boxes", "cardinality"]
    ref = criterion_oracle.SetCriterion(NUM_CLASSES, criterion_oracle.HungarianMatcher(2, 5, 2), WEIGHTS, losses)
    crit = dfvod_b200.SetCriterion(NUM_CLASSES, dfvod_b200.HungarianMatcher(2, 5, 2), WEIGHTS, losses)
    padded = dfvod_b200.pad_targets(targets, 30)
    run = lambda: model(srcs, masks, poss, dsrcs, dmasks, dposs, query)
    opt = torch.optim.AdamW(model.parameters(), lr=1e-5, fused=True)

    def eager():
        opt.zero_grad(set_to_none=True)
        loss = weighted(ref(run(), targets))
        loss.backward()
        opt.step()
        return loss

    model2 = copy.deepcopy(model)
    opt2 = torch.optim.AdamW(model2.parameters(), lr=1e-5, fused=True)
    run2 = lambda: model2(srcs, masks, poss, dsrcs, dmasks, dposs, query)
    eager_loss = float(eager().detach())
    eager()
    step = data_parallel.GraphedTrainStep(model2, opt2, lambda: weighted(crit(run2(), padded)))
    graphed_loss = float(step().detach())
    print(f"first-step loss: eager reference-form {eager_loss:.6f}, graphed {graphed_loss:.6f}", flush=True)
    fns = {"graphed, SetCriterion (padded)": step, "eager, reference-form criterion": eager}
    times = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            times[k].append(timed(fn, step_iters))
    for k, v in times.items():
        print(f"C5 Encoder-CF training step with the criterion, bf16, 4 frames, {k}: {statistics.median(v):.2f} ms "
              f"(spread {min(v):.2f}-{max(v):.2f})", flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--step-iters", type=int, default=5)
    ap.add_argument("--no-step", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_criterion.py needs a CUDA device")
    print(card(), flush=True)
    matcher(args.iters, args.rounds)
    if not args.no_step:
        train_step(args.step_iters, args.rounds)


if __name__ == "__main__":
    main()
