"""GPU: the batched linear-assignment kernel (csrc/hungarian.cu) against scipy, and dfvod_b200.criterion against the
reference restated in oracle/criterion_oracle.py: matcher pairs, losses and gradients, no host sync, and a graphed
training step on the real criterion against the eager reference-form loop."""
import copy

import numpy as np
import pytest
import torch
from scipy.optimize import linear_sum_assignment

import dfvod_b200
from dfvod_b200 import criterion, data_parallel
from oracle import criterion_oracle

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def solve(cost, counts):
    m = criterion.linear_assignment(cost, torch.as_tensor(counts, dtype=torch.int64, device=DEV))
    return [x.cpu() for x in m]


def check_optimal(cost, counts, qot, toq, status, identical):
    """Every problem solved; the matching is one-to-one and covers the targets; with `identical` it is scipy's,
    otherwise its total cost is scipy's optimum."""
    cost = cost.double().cpu().numpy()
    for p, n in enumerate(counts):
        assert int(status[p]) == 0, p
        rows, cols = linear_sum_assignment(cost[p, :, :n])
        q_of_t = qot[p].numpy()
        assert (q_of_t[n:] == -1).all()
        t_of_q = toq[p].numpy()
        assert (t_of_q >= 0).sum() == n and (t_of_q < n).all()
        if n:
            assert len(set(q_of_t[:n].tolist())) == n and (q_of_t[:n] >= 0).all()
            assert (t_of_q[q_of_t[:n]] == np.arange(n)).all(), p
        if identical:
            want = np.full(cost.shape[1], -1)
            want[rows] = cols
            assert (t_of_q == want).all(), p
        else:
            got = cost[p, q_of_t[:n], np.arange(n)].sum()
            assert got == cost[p, rows, cols].sum(), (p, got, cost[p, rows, cols].sum())


SOLVER_CASES = [(1, 64), (17, 64), (300, 64), (1000, 16), (4200, 4), (22223, 3)]


@pytest.mark.parametrize("q,problems", SOLVER_CASES)
def test_solver_matches_scipy_on_continuous_costs(q, problems):
    g = torch.Generator().manual_seed(q)
    sizes = [t for t in (0, 1, 5, 100) if t <= q] + ([q] if q <= 300 else [])
    counts = [sizes[(p * 7 + 3) % len(sizes)] for p in range(problems)]
    tmax = max(counts)
    # a strided view: the query stride (tmax + 3) is not the number of target slots
    big = torch.randn(problems, q, tmax + 3, generator=g).to(DEV)
    cost = big[:, :, :tmax]
    qot, toq, status = solve(cost, counts)
    check_optimal(cost, counts, qot, toq, status, identical=True)


@pytest.mark.parametrize("q", [17, 300, 1500])
def test_solver_is_optimal_on_tied_costs(q):
    g = torch.Generator().manual_seed(5)
    counts = [min(q, t) for t in (1, 5, 17, 100, 0, 9)]
    tmax = max(counts)
    ints = torch.randint(0, 4, (6, q, tmax), generator=g).float()
    ints[4:] = 2.5                         # all-equal costs
    cost = ints.to(DEV)
    qot, toq, status = solve(cost, counts)
    check_optimal(cost, counts, qot, toq, status, identical=False)


@pytest.mark.parametrize("q", [300, 4200])
def test_solver_flags_nonfinite_costs_and_bad_counts(q):
    g = torch.Generator().manual_seed(9)
    counts = [5, 5, 5, 5, 7, 6, -1, 5]       # 7 is above the 6 target slots, -1 below zero
    cost = torch.rand(8, q, 6, generator=g)
    cost[0, q // 2, 4] = float("nan")
    cost[1, 0, 0] = float("inf")
    cost[2, q - 1, 2] = -float("inf")
    cost[3, 3, 5] = float("nan")            # beyond the problem's 5 targets: not read
    cost = cost.to(DEV)
    qot, toq, status = solve(cost, counts)
    assert status.tolist() == [1, 1, 1, 0, 2, 0, 2, 0]
    for p in (0, 1, 2, 4, 6):
        assert (qot[p] == -1).all() and (toq[p] == -1).all()
    ok = [3, 5, 7]
    check_optimal(cost[ok], [counts[p] for p in ok], qot[ok], toq[ok], status[ok], identical=True)


def deformable_outputs(seed, b=4, q=300, k=91, layers=6, counts=(0, 7, 40, 100), enc_q=None, dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)

    def head(nq):
        return {"pred_logits": (torch.randn(b, nq, k, generator=g) * 2 - 3).to(DEV, dtype).requires_grad_(True),
                "pred_boxes": torch.randn(b, nq, 4, generator=g).mul(1.2).sigmoid().to(DEV, dtype)
                .requires_grad_(True)}

    outputs = head(q)
    outputs["aux_outputs"] = [head(q) for _ in range(layers - 1)]
    if enc_q:
        outputs["enc_outputs"] = head(enc_q)
    targets = []
    for n in counts:
        cxcy = torch.rand(n, 2, generator=g) * 0.8 + 0.1
        wh = torch.rand(n, 2, generator=g) * 0.3 + 0.01
        targets.append({"labels": torch.randint(0, k, (n,), generator=g).to(DEV),
                        "boxes": torch.cat([cxcy, wh], 1).to(DEV, dtype)})
    return outputs, targets


def heads_of(outputs):
    return [outputs] + outputs.get("aux_outputs", []) + ([outputs["enc_outputs"]] if "enc_outputs" in outputs else [])


@pytest.mark.parametrize("num_classes", [2, 31, 91])
def test_matcher_pairs_are_the_reference_pairs(num_classes):
    outputs, targets = deformable_outputs(num_classes, k=num_classes)
    mine, ref = dfvod_b200.HungarianMatcher(2, 5, 2), criterion_oracle.HungarianMatcher(2, 5, 2)
    for h in heads_of(outputs):
        got = mine(h, targets)
        want = ref(h, targets)                # the reference: fp32 cost on the GPU, scipy on the CPU
        for (gi, gj), (wi, wj) in zip(got, want):
            assert gi.device == DEV and gi.dtype == torch.int64 and gj.dtype == torch.int64
            assert torch.equal(gi.cpu(), wi) and torch.equal(gj.cpu(), wj)


def to_fp64_cpu(outputs):
    return {k: ([to_fp64_cpu(a) for a in v] if k == "aux_outputs" else
                to_fp64_cpu(v) if k == "enc_outputs" else v.detach().double().cpu().requires_grad_(True))
            for k, v in outputs.items()}


def nerr(x, ref):
    x, ref = x.double().cpu(), ref.double().cpu()
    scale = ref.abs().max().clamp_min(1e-30)
    return float((x - ref).abs().max() / scale), float((x - ref).norm() / ref.norm().clamp_min(1e-30))


WEIGHTS = {"loss_ce": 2.0, "loss_bbox": 5.0, "loss_giou": 2.0}


def weighted(losses):
    base = lambda k: k if k in WEIGHTS else k.rsplit("_", 1)[0]
    return sum(v * WEIGHTS[base(k)] for k, v in losses.items() if base(k) in WEIGHTS)


@pytest.mark.parametrize("layers,enc_q", [(1, None), (6, None), (6, 1200)])
def test_criterion_matches_the_fp64_oracle(layers, enc_q):
    outputs, targets = deformable_outputs(11 + layers, layers=layers, enc_q=enc_q, counts=(3, 0, 30, 100))
    ref_out = to_fp64_cpu(outputs)
    ref_targets = [{k: v.double().cpu() if v.is_floating_point() else v.cpu() for k, v in t.items()} for t in targets]
    losses = ["labels", "boxes", "cardinality"]
    crit = dfvod_b200.SetCriterion(91, dfvod_b200.HungarianMatcher(2, 5, 2), WEIGHTS, losses)
    ref = criterion_oracle.SetCriterion(91, criterion_oracle.HungarianMatcher(2, 5, 2), WEIGHTS, losses)
    for form in ("list", "padded"):
        got = crit(outputs, targets if form == "list" else dfvod_b200.pad_targets(targets, 100))
        want = ref(ref_out, ref_targets)
        assert sorted(got) == sorted(want)
        for k, w in want.items():
            g = float(got[k])
            assert abs(g - float(w)) <= 1e-6 * abs(float(w)) + 1e-7, (form, k, g, float(w))
        mine = torch.autograd.grad(weighted(got), [h[n] for h in heads_of(outputs) for n in ("pred_logits", "pred_boxes")])
        theirs = torch.autograd.grad(weighted(want), [h[n] for h in heads_of(ref_out) for n in ("pred_logits", "pred_boxes")])
        for i, (a, b) in enumerate(zip(mine, theirs)):
            mx, l2 = nerr(a, b)
            assert mx <= 1e-5 and l2 <= 1e-5, (form, i, mx, l2)


def test_padded_criterion_does_not_sync():
    outputs, targets = deformable_outputs(21, enc_q=1200)
    padded = dfvod_b200.pad_targets(targets, 100)
    crit = dfvod_b200.SetCriterion(91, dfvod_b200.HungarianMatcher(2, 5, 2), WEIGHTS, ["labels", "boxes", "cardinality"])
    leaves = [h[n] for h in heads_of(outputs) for n in ("pred_logits", "pred_boxes")]
    for _ in range(2):
        torch.autograd.grad(weighted(crit(outputs, padded)), leaves)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        grads = torch.autograd.grad(weighted(crit(outputs, padded)), leaves)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert all(bool(torch.isfinite(g).all()) for g in grads)


def inverse_sigmoid(x, eps=1e-5):
    x = x.clamp(min=0, max=1)
    return torch.log(x.clamp(min=eps) / (1 - x).clamp(min=eps))


class Detector(torch.nn.Module):
    """Deformable DETR's heads (single-scale class head, 3-layer box MLP, no box refinement) on the package's
    transformer: test-side, as in the reference's DeformableDETR.forward."""

    def __init__(self, num_classes, num_queries=60):
        super().__init__()
        from dfvod_b200.deformable_transformer import DeformableTransformer
        self.transformer = DeformableTransformer(num_encoder_layers=2, num_decoder_layers=2, num_feature_levels=2,
                                                 dropout=0.0, return_intermediate_dec=True)
        self.class_embed = torch.nn.Linear(256, num_classes)
        self.bbox_embed = torch.nn.Sequential(torch.nn.Linear(256, 256), torch.nn.ReLU(), torch.nn.Linear(256, 256),
                                              torch.nn.ReLU(), torch.nn.Linear(256, 4))
        self.query_embed = torch.nn.Embedding(num_queries, 512)

    def forward(self, srcs, masks, poss):
        hs, init_ref, inter_refs, _, _ = self.transformer(srcs, masks, poss, None, None, None, self.query_embed.weight)
        classes, coords = [], []
        for lvl in range(hs.shape[0]):
            reference = inverse_sigmoid(init_ref if lvl == 0 else inter_refs[lvl - 1])
            tmp = self.bbox_embed(hs[lvl])
            coords.append(torch.cat([tmp[..., :2] + reference, tmp[..., 2:]], -1).sigmoid())
            classes.append(self.class_embed(hs[lvl]))
        return {"pred_logits": classes[-1], "pred_boxes": coords[-1],
                "aux_outputs": [{"pred_logits": a, "pred_boxes": b} for a, b in zip(classes[:-1], coords[:-1])]}


def test_graphed_step_with_the_real_criterion_matches_the_eager_reference():
    torch.manual_seed(2)
    num_classes, tmax = 5, 12
    shapes = [(12, 16), (6, 8)]
    model = Detector(num_classes).to(DEV)
    with torch.no_grad():                 # off the zero-initialised sampling offsets, as test_gpu_graphed_step.py
        for p in model.parameters():
            p.add_(torch.randn_like(p) * 0.02)
    model2 = copy.deepcopy(model)
    srcs = [torch.randn(2, 256, h, w, device=DEV) for h, w in shapes]
    poss = [torch.randn(2, 256, h, w, device=DEV) for h, w in shapes]
    masks = [torch.zeros(2, h, w, dtype=torch.bool, device=DEV) for h, w in shapes]
    g = torch.Generator().manual_seed(8)

    def batch(counts):
        return [{"labels": torch.randint(0, num_classes, (n,), generator=g).to(DEV),
                 "boxes": torch.cat([torch.rand(n, 2, generator=g) * 0.8 + 0.1,
                                     torch.rand(n, 2, generator=g) * 0.3 + 0.05], 1).to(DEV)} for n in counts]

    batches = [batch((3, 9)), batch((0, 12)), batch((7, 1))]
    losses = ["labels", "boxes", "cardinality"]
    ref = criterion_oracle.SetCriterion(num_classes, criterion_oracle.HungarianMatcher(2, 5, 2), WEIGHTS, losses)
    crit = dfvod_b200.SetCriterion(num_classes, dfvod_b200.HungarianMatcher(2, 5, 2), WEIGHTS, losses)

    opt = torch.optim.SGD(model.parameters(), lr=0.01)
    eager = []
    for targets in batches:
        opt.zero_grad(set_to_none=True)
        loss = weighted(ref(model(srcs, masks, poss), targets))
        loss.backward()
        opt.step()
        eager.append(float(loss))

    static = dfvod_b200.pad_targets(batches[0], tmax)
    opt2 = torch.optim.SGD(model2.parameters(), lr=0.01)
    step = data_parallel.GraphedTrainStep(model2, opt2, lambda: weighted(crit(model2(srcs, masks, poss), static)))
    graphed = []
    for targets in batches:
        for dst, src in zip(static, dfvod_b200.pad_targets(targets, tmax)):
            dst.copy_(src)
        graphed.append(float(step()))
    torch.cuda.synchronize()
    for a, b in zip(eager, graphed):
        assert abs(a - b) <= 1e-5 * abs(a), (eager, graphed)
    for (name, p), q in zip(model.named_parameters(), model2.parameters()):
        err = float((p - q).abs().max() / p.abs().max().clamp_min(1e-12))
        assert err <= 2e-5, (name, err)
