"""CPU: dfvod_b200.criterion's host composition.  pad_targets packs and validates; with the device solver replaced
by scipy (oracle side only, as test_host_logic_cpu.py replaces the attention op) the matcher returns the reference's
pairs and SetCriterion reproduces oracle/criterion_oracle.py's losses and gradients in fp64."""
import numpy as np
import pytest
import torch
from scipy.optimize import linear_sum_assignment

import dfvod_b200
from dfvod_b200 import criterion
from oracle import criterion_oracle


def scipy_assignment(cost, counts):
    """linear_assignment's contract, solved by scipy per problem."""
    p, q, t = cost.shape
    qot = torch.full((p, t), -1, dtype=torch.int32)
    toq = torch.full((p, q), -1, dtype=torch.int32)
    status = torch.zeros(p, dtype=torch.int32)
    for k in range(p):
        n = int(counts[k])
        c = cost[k, :, :n].detach().double().numpy()
        if not np.isfinite(c).all():
            status[k] = 1
            continue
        rows, cols = linear_sum_assignment(c)
        qot[k, torch.as_tensor(cols)] = torch.as_tensor(rows, dtype=torch.int32)
        toq[k, torch.as_tensor(rows)] = torch.as_tensor(cols, dtype=torch.int32)
    return criterion.Matching(qot, toq, status)


@pytest.fixture()
def scipy_solver(monkeypatch):
    monkeypatch.setattr(criterion, "linear_assignment", scipy_assignment)


def make_batch(seed, b=3, q=40, k=7, layers=3, counts=(5, 0, 12), enc_q=None, dtype=torch.float64):
    g = torch.Generator().manual_seed(seed)
    mk = lambda *s: torch.randn(*s, generator=g, dtype=dtype)

    def head(nq):
        return {"pred_logits": mk(b, nq, k).requires_grad_(True),
                "pred_boxes": (mk(b, nq, 4) * 0.8).sigmoid().requires_grad_(True)}

    outputs = head(q)
    outputs["aux_outputs"] = [head(q) for _ in range(layers - 1)]
    if enc_q:
        outputs["enc_outputs"] = head(enc_q)
    targets = []
    for n in counts:
        cxcy = torch.rand(n, 2, generator=g, dtype=dtype) * 0.8 + 0.1
        wh = torch.rand(n, 2, generator=g, dtype=dtype) * 0.3 + 0.02
        targets.append({"labels": torch.randint(0, k, (n,), generator=g), "boxes": torch.cat([cxcy, wh], 1)})
    return outputs, targets


def leaves(outputs):
    heads = [outputs] + outputs.get("aux_outputs", []) + ([outputs["enc_outputs"]] if "enc_outputs" in outputs else [])
    return [h[name] for h in heads for name in ("pred_logits", "pred_boxes")]


def test_pad_targets_packs_and_pads_with_a_valid_box():
    _, targets = make_batch(0)
    p = dfvod_b200.pad_targets(targets, 16)
    assert p.labels.shape == (3, 16) and p.boxes.shape == (3, 16, 4) and p.counts.tolist() == [5, 0, 12]
    assert p.labels.dtype == torch.int64 and p.counts.dtype == torch.int64 and p.boxes.dtype == torch.float64
    for b, t in enumerate(targets):
        n = len(t["labels"])
        assert torch.equal(p.labels[b, :n], t["labels"]) and torch.equal(p.boxes[b, :n], t["boxes"])
        assert not p.labels[b, n:].any()
        assert torch.equal(p.boxes[b, n:], torch.tensor([0.5, 0.5, 1.0, 1.0], dtype=torch.float64).expand(16 - n, 4))


def test_pad_targets_rejects_malformed_input():
    _, targets = make_batch(0)
    with pytest.raises(ValueError, match="more than max_boxes"):
        dfvod_b200.pad_targets(targets, 11)
    with pytest.raises(ValueError, match="at least 1"):
        dfvod_b200.pad_targets(targets, 0)
    with pytest.raises(ValueError, match="at least one image"):
        dfvod_b200.pad_targets([], 4)
    bad = [dict(t) for t in targets]
    bad[0]["labels"] = bad[0]["labels"].float()
    with pytest.raises(ValueError, match="1-D integer"):
        dfvod_b200.pad_targets(bad, 16)
    bad = [dict(t) for t in targets]
    bad[2]["boxes"] = bad[2]["boxes"][:, :3]
    with pytest.raises(ValueError, match=r"floating \[12, 4\]"):
        dfvod_b200.pad_targets(bad, 16)
    bad = [dict(t) for t in targets]
    bad[0]["boxes"] = bad[0]["boxes"][:4]
    with pytest.raises(ValueError, match=r"\[5, 4\]"):
        dfvod_b200.pad_targets(bad, 16)
    bad = [dict(t) for t in targets]
    bad[0]["labels"] = bad[0]["labels"].clone()
    bad[0]["labels"][1] = -1
    with pytest.raises(ValueError, match="negative label"):
        dfvod_b200.pad_targets(bad, 16)
    for value, col in ((float("nan"), 0), (float("inf"), 1), (-0.1, 2)):
        bad = [dict(t) for t in targets]
        bad[2]["boxes"] = bad[2]["boxes"].clone()
        bad[2]["boxes"][3, col] = value
        with pytest.raises(ValueError, match="finite with non-negative"):
            dfvod_b200.pad_targets(bad, 16)


def test_more_target_slots_than_queries_is_rejected(scipy_solver):
    outputs, targets = make_batch(1, q=10, counts=(3, 4, 2))
    crit = dfvod_b200.SetCriterion(7, dfvod_b200.HungarianMatcher(), {}, ["labels", "boxes"])
    with pytest.raises(ValueError, match="11 target slots for 10 queries"):
        crit(outputs, dfvod_b200.pad_targets(targets, 11))
    with pytest.raises(ValueError, match="13 target slots for 10 queries"):
        dfvod_b200.HungarianMatcher()(outputs, targets + [{"labels": torch.zeros(13, dtype=torch.int64),
                                                            "boxes": torch.full((13, 4), 0.2, dtype=torch.float64)}])


def test_linear_assignment_refuses_cpu_tensors():
    with pytest.raises(RuntimeError, match="Not implemented on the CPU"):
        criterion.linear_assignment(torch.zeros(2, 5, 3), torch.tensor([3, 1]))


@pytest.mark.parametrize("weights", [(1, 1, 1), (2, 5, 2)])
def test_matcher_pairs_match_the_oracle(scipy_solver, weights):
    outputs, targets = make_batch(2, b=4, counts=(5, 0, 12, 40))
    got = dfvod_b200.HungarianMatcher(*weights)(outputs, targets)
    want = criterion_oracle.HungarianMatcher(*weights)(outputs, targets)
    assert len(got) == len(want) == 4
    for (gi, gj), (wi, wj) in zip(got, want):
        assert gi.dtype == gj.dtype == torch.int64
        assert torch.equal(gi, wi) and torch.equal(gj, wj)


@pytest.mark.parametrize("enc_q", [None, 60])
@pytest.mark.parametrize("form", ["list", "padded"])
def test_criterion_reproduces_the_oracle_in_fp64(scipy_solver, enc_q, form):
    outputs, targets = make_batch(3, enc_q=enc_q)
    weight_dict = {"loss_ce": 2.0, "loss_bbox": 5.0, "loss_giou": 2.0}
    losses = ["labels", "boxes", "cardinality"]
    crit = dfvod_b200.SetCriterion(7, dfvod_b200.HungarianMatcher(2, 5, 2), weight_dict, losses)
    ref = criterion_oracle.SetCriterion(7, criterion_oracle.HungarianMatcher(2, 5, 2), weight_dict, losses)
    got = crit(outputs, targets if form == "list" else dfvod_b200.pad_targets(targets, 20))
    want = ref(outputs, targets)
    assert sorted(got) == sorted(want)
    assert "class_error" in got and "loss_ce_1" in got and ("loss_giou_enc" in got) == bool(enc_q)
    for k in want:
        assert got[k].dtype == want[k].dtype, k
        np.testing.assert_allclose(float(got[k]), float(want[k]), rtol=1e-12, atol=1e-12, err_msg=k)

    def grads(d):
        base = lambda k: k if k in weight_dict else k.rsplit("_", 1)[0]
        total = sum(d[k] * weight_dict[base(k)] for k in d if base(k) in weight_dict)
        return torch.autograd.grad(total, leaves(outputs))

    for g, w in zip(grads(got), grads(want)):
        np.testing.assert_allclose(g.numpy(), w.numpy(), rtol=1e-10, atol=1e-14)


def test_criterion_without_boxes_and_with_given_num_boxes(scipy_solver):
    outputs, targets = make_batch(4, counts=(0, 0, 0))
    crit = dfvod_b200.SetCriterion(7, dfvod_b200.HungarianMatcher(), {}, ["labels", "boxes", "cardinality"])
    ref = criterion_oracle.SetCriterion(7, criterion_oracle.HungarianMatcher(), {}, ["labels", "boxes",
                                                                                    "cardinality"])
    got, want = crit(outputs, targets), ref(outputs, targets)
    for k in want:
        np.testing.assert_allclose(float(got[k]), float(want[k]), rtol=1e-12, atol=1e-12, err_msg=k)
    assert float(got["class_error"]) == 100.0 and float(got["loss_bbox"]) == 0.0
    outputs, targets = make_batch(5)
    a = crit(outputs, targets)
    b = crit(outputs, targets, num_boxes=2 * 17)
    for k in ("loss_ce", "loss_bbox", "loss_giou_1"):
        np.testing.assert_allclose(float(b[k]) * 2, float(a[k]), rtol=1e-12, err_msg=k)


def test_nonfinite_cost_poisons_only_its_head(scipy_solver):
    outputs, targets = make_batch(6)
    with torch.no_grad():
        outputs["aux_outputs"][1]["pred_boxes"][2, 7, 0] = float("nan")
    crit = dfvod_b200.SetCriterion(7, dfvod_b200.HungarianMatcher(), {}, ["labels", "boxes"])
    got = crit(outputs, dfvod_b200.pad_targets(targets, 12))
    for k, v in got.items():
        assert bool(torch.isnan(v)) == k.endswith("_1"), k
    (got["loss_ce_1"] + got["loss_bbox"]).backward()
    assert torch.isnan(outputs["aux_outputs"][1]["pred_logits"].grad).all()
    assert torch.isfinite(outputs["pred_boxes"].grad).all()


def test_unsupported_loss_is_refused():
    with pytest.raises(ValueError, match="masks"):
        dfvod_b200.SetCriterion(7, dfvod_b200.HungarianMatcher(), {}, ["labels", "masks"])
