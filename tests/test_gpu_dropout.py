"""GPU: dropout on the package's kernels (DESIGN.md section 3.16) against the numpy Philox oracle (tests/philox_oracle.py).

Every mask is checked bit for bit: the key each call draws is recorded (layer_epilogue_func._dropout_key is wrapped),
the oracle rebuilds the mask from it, and the reference is a torch composition in fp64 with that mask.  Tolerances are
those of tests/test_gpu_layer_epilogue.py (add-LayerNorm) and of the linear training tests; a wrong mask would be off
by O(1)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from torch import nn

from dfvod_b200 import _lib
from dfvod_b200.ops.functions import layer_epilogue_func as lef

from .philox_oracle import keep_mask, rule

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = {torch.float32: 1e-5, torch.bfloat16: 2.0 ** -7, torch.float16: 2.0 ** -9}
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def nerr(x, ref):
    x, ref = x.detach().double(), ref.detach().double()
    return float((x - ref).abs().max() / ref.abs().max().clamp_min(1e-300))


@pytest.fixture
def keys(monkeypatch):
    drawn = []
    real = lef._dropout_key

    def record(device):
        k = real(device)
        drawn.append(k)
        return k
    monkeypatch.setattr(lef, "_dropout_key", record)
    return drawn


def oracle_mask(key, shape, p, device=DEV):
    n = int(np.prod(shape))
    return torch.from_numpy(keep_mask(int(key.item()), n, p)).to(device).view(shape)


def train_dropout(p):
    return nn.Dropout(p).train()


# ---------------------------------------------------------------------------------------------------------------------
# mask exactness
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("n", [8, 13, 4096 + 5, 1_000_003])
@pytest.mark.parametrize("p", [0.1, 0.5])
def test_dropout_mask_is_the_oracle_mask(keys, dtype, n, p):
    x = torch.ones(n, dtype=dtype, device=DEV, requires_grad=True)
    y = lef.dropout(train_dropout(p), x)
    assert len(keys) == 1
    m = oracle_mask(keys[0], (n,), p)
    scale = rule(p)[1]
    assert torch.equal(y, (m.float() * scale).to(dtype))
    y.backward(torch.ones_like(y))                       # the backward regenerates the same mask
    assert torch.equal(x.grad, (m.float() * scale).to(dtype))


def test_dropout_in_place_and_unaligned():
    key = torch.tensor([123456789], dtype=torch.int64, device=DEV)
    buf = torch.ones(1001, device=DEV)
    x = buf[1:]                                        # 4-byte offset: the element-by-element path
    lef._dropout_into(x, x, 0.2, key)
    m = oracle_mask(key, (1000,), 0.2)
    assert torch.equal(x, m.float() * rule(0.2)[1]) and buf[0] == 1


def test_refusals():
    lib = _lib.load()
    key = torch.zeros(1, dtype=torch.int64, device=DEV)
    x = torch.ones(64, device=DEV)
    for p in (0.0, 1.0, -0.5, float("nan")):
        assert lib.msda_layer_dropout(_lib.DTYPE_F32, x.data_ptr(), x.data_ptr(), 64, p, key.data_ptr(), 0) != 0
    assert lib.msda_layer_dropout(_lib.DTYPE_F32, x.data_ptr(), x.data_ptr(), 64, 0.1, None, 0) != 0
    assert lib.msda_layer_linear_bf16_relu_dropout(None, None, None, 256, 256, 256, 0.1, None, None, 0) != 0
    assert not lib.msda_layer_add_layernorm_dropout_supported(_lib.DTYPE_BF16, 1024)


# ---------------------------------------------------------------------------------------------------------------------
# add-LayerNorm with dropout
def ref_chain(norm64, branch, residual, act, pos, mask, scale):
    h = branch.double()
    if act == "relu":
        h = F.relu(h)
    elif act == "gelu":
        h = F.gelu(h)
    h = h * mask.double() * scale
    v = h if residual is None else residual.double() + h
    y = norm64(v)
    return y, (None if pos is None else y + pos.double())


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("act", [None, "relu", "gelu"])
@pytest.mark.parametrize("with_res,with_pos", [(True, True), (True, False), (False, False)])
def test_add_layer_norm_dropout_forward_backward(keys, dtype, act, with_res, with_pos):
    c, p = 256, 0.2
    torch.manual_seed(7)
    rows = (3, 347)
    norm = nn.LayerNorm(c).to(DEV)
    with torch.no_grad():
        norm.weight.add_(torch.randn(c, device=DEV) * 0.3)
        norm.bias.add_(torch.randn(c, device=DEV) * 0.3)
    norm = norm.to(dtype)
    norm64 = nn.LayerNorm(c).to(DEV).double()
    norm64.load_state_dict({k: v.double() for k, v in norm.state_dict().items()})
    mk = lambda: (torch.randn(*rows, c, device=DEV) * 1.5).to(dtype)
    leaves = [mk().requires_grad_(True) for _ in range(1 + with_res + with_pos)]
    b = leaves[0]
    r = leaves[1] if with_res else None
    q = leaves[-1] if with_pos else None
    out = lef.add_layer_norm(norm, b, r, act, q, dropout=train_dropout(p))
    assert len(keys) == 1
    y, y_pos = out if with_pos else (out, None)
    mask = oracle_mask(keys[0], b.shape, p)
    leaves64 = [t.detach().double().requires_grad_(True) for t in leaves]
    b64 = leaves64[0]
    r64 = leaves64[1] if with_res else None
    q64 = leaves64[-1] if with_pos else None
    y64, y_pos64 = ref_chain(norm64, b64, r64, act, q64, mask, rule(p)[1])
    tol = TOL[dtype]
    assert nerr(y, y64) <= tol
    if with_pos:
        assert nerr(y_pos, y_pos64) <= tol
    gy = torch.randn_like(y)
    gyp = torch.randn_like(y) if with_pos else None
    ((y.float() * gy.float()).sum() + ((y_pos.float() * gyp.float()).sum() if with_pos else 0)).backward()
    ((y64 * gy.double()).sum() + ((y_pos64 * gyp.double()).sum() if with_pos else 0)).backward()
    gtol = tol * 4 if dtype != torch.float32 else 2e-5
    for a, ref in zip(leaves, leaves64):
        assert nerr(a.grad, ref.grad) <= gtol
    assert nerr(norm.weight.grad, norm64.weight.grad) <= gtol
    assert nerr(norm.bias.grad, norm64.bias.grad) <= gtol


# ---------------------------------------------------------------------------------------------------------------------
# ReLU -> dropout linear on the bf16-kernel, tf32x3-kernel and library routes
ROUTES = {"bf16_kernel": (torch.bfloat16, "library", 16384, 2.0 ** -7),
          "tf32x3_kernel": (torch.float32, "tf32x3", 2400, 1e-5),
          "library_fp32": (torch.float32, "library", 2400, 1e-5),
          "library_bf16": (torch.bfloat16, "library", 1000, 2.0 ** -7)}


@pytest.mark.parametrize("route", list(ROUTES))
def test_linear_relu_dropout_routes(keys, monkeypatch, route):
    dtype, mode, rows, tol = ROUTES[route]
    monkeypatch.setattr(lef, "FP32_TRAIN_GEMM_MODE", mode)
    torch.manual_seed(3)
    n, k, p = 1024, 256, 0.1
    lin = nn.Linear(k, n).to(DEV).to(dtype)
    x = torch.randn(rows, k, device=DEV).to(dtype).requires_grad_(True)
    y = lef.linear_relu(lin, x, train_dropout(p))
    assert len(keys) == 1
    mask = oracle_mask(keys[0], (rows, n), p)
    assert bool((y[~mask] == 0).all())
    x64 = x.detach().double().requires_grad_(True)
    w64 = lin.weight.detach().double().requires_grad_(True)
    b64 = lin.bias.detach().double().requires_grad_(True)
    y64 = F.relu(x64 @ w64.t() + b64) * mask.double() * rule(p)[1]
    assert nerr(y, y64) <= 4 * tol
    g = torch.randn_like(y)
    y.backward(g)
    y64.backward(g.double())
    for a, ref in ((x.grad, x64.grad), (lin.weight.grad, w64.grad), (lin.bias.grad, b64.grad)):
        assert nerr(a, ref) <= 8 * tol


@pytest.mark.parametrize("kind", ["bf16", "tf32x3"])
def test_relu_dropout_gemm_writes_only_y(kind):
    torch.manual_seed(5)
    rows, n, k, p = 3000, 256, 256, 0.3
    dt = torch.bfloat16 if kind == "bf16" else torch.float32
    x = torch.randn(rows, k, device=DEV).to(dt)
    w = (torch.randn(n, k, device=DEV) * 0.05).to(dt)
    b = torch.randn(n, device=DEV).to(dt)
    key = torch.tensor([-987654321987], dtype=torch.int64, device=DEV)
    guard = 4096
    buf = torch.full((rows * n + 2 * guard,), float("nan"), device=DEV).to(dt)
    y = buf[guard:guard + rows * n].view(rows, n)
    lib = _lib.load()
    if kind == "bf16":
        code = lib.msda_layer_linear_bf16_relu_dropout(x.data_ptr(), w.data_ptr(), b.data_ptr(), rows, n, k, p,
                                                       key.data_ptr(), y.data_ptr(), 0)
    else:
        w_hi, w_lo = lef._tf32_weight_split(w)
        code = lib.msda_layer_linear_tf32x3_relu_dropout(x.data_ptr(), w_hi.data_ptr(), w_lo.data_ptr(), b.data_ptr(),
                                                         rows, n, k, p, key.data_ptr(), y.data_ptr(), 0)
    torch.cuda.synchronize()
    assert code == 0
    assert bool(buf[:guard].isnan().all()) and bool(buf[guard + rows * n:].isnan().all())
    mask = oracle_mask(key, (rows, n), p)
    ref = F.relu(x.double() @ w.double().t() + b.double()) * mask.double() * rule(p)[1]
    assert bool((y[~mask] == 0).all())
    assert nerr(y, ref) <= (2.0 ** -7 if kind == "bf16" else 1e-5) * 4


# ---------------------------------------------------------------------------------------------------------------------
# statistics
def test_keep_rate_and_independence():
    p = 0.1
    t = rule(p)[0]
    q = 1 - t / 65536
    n = 1 << 26
    key = torch.tensor([42], dtype=torch.int64, device=DEV)
    ones = torch.ones(n, device=DEV)
    m = lef._dropout_into(ones, torch.empty_like(ones), p, key) != 0
    rate = float(m.double().mean())
    assert abs(rate - q) <= 6 * (q * (1 - q) / n) ** 0.5
    rows, cols = n // 1024, 1024
    mm = m.view(rows, cols).double()
    col = mm.mean(0)
    row = mm.mean(1)
    assert float((col - q).abs().max()) <= 6 * (q * (1 - q) / rows) ** 0.5
    assert float((row - q).abs().max()) <= 6 * (q * (1 - q) / cols) ** 0.5 + 1e-12
    # successive calls draw fresh keys: their masks are uncorrelated
    a = lef.dropout(train_dropout(p), ones[: 1 << 24]) != 0
    b = lef.dropout(train_dropout(p), ones[: 1 << 24]) != 0
    a, b = a.double() - a.double().mean(), b.double() - b.double().mean()
    corr = float((a * b).mean() / (a.std() * b.std()))
    assert abs(corr) <= 6 / (1 << 12)


# ---------------------------------------------------------------------------------------------------------------------
# reproducibility and the paths that draw no key
def test_same_seed_same_bits_other_seed_other_bits():
    norm = nn.LayerNorm(256).to(DEV).bfloat16()
    x = torch.randn(5000, 256, device=DEV).bfloat16()

    def run(seed):
        torch.manual_seed(seed)
        b = x.clone().requires_grad_(True)
        y = lef.add_layer_norm(norm, b, x, "gelu", dropout=train_dropout(0.1))
        y.float().square().sum().backward()
        return y.detach(), b.grad
    y1, g1 = run(1)
    y2, g2 = run(1)
    y3, g3 = run(2)
    assert torch.equal(y1, y2) and torch.equal(g1, g2)
    assert not torch.equal(y1, y3) and not torch.equal(g1, g3)


def test_no_key_at_p0_or_eval_and_torch_at_p1(keys):
    norm = nn.LayerNorm(256).to(DEV)
    x = torch.randn(300, 256, device=DEV)
    plain = lef.add_layer_norm(norm, x, x, "gelu")
    for module in (nn.Dropout(0.0).train(), nn.Dropout(0.1).eval()):
        state = torch.cuda.get_rng_state()
        assert torch.equal(lef.add_layer_norm(norm, x, x, "gelu", dropout=module), plain)
        assert torch.equal(torch.cuda.get_rng_state(), state)
    assert not keys
    # p = 1: torch's nn.Dropout drops everything
    y = lef.add_layer_norm(norm, x, x, "gelu", dropout=nn.Dropout(1.0).train())
    assert not keys
    assert torch.allclose(y, norm(x), atol=1e-5)


# ---------------------------------------------------------------------------------------------------------------------
# layers in train() at p = 0.1 against the fp64 torch composition with the recorded masks
LAYERS = ["layer_encoder_c256", "layer_fusion_v2_c256", "layer_late_fusion_c256", "decoder_c128",
          "backbone_udf_fuse_c128"]
FP32_LAYER_TOL = 1e-4
LOOSE = ("pos", "query_pos", "sampling_offsets", "attention_weights")


def _within_layer_bounds(dtype, name, x, ref):
    """fp32: normalised max error 1e-4.  bf16: the relative-L2 layer bounds of
    tests/test_gpu_linear_bf16_train.py::test_layers_train_on_the_kernels_within_bf16_bounds (output 2^-6, gradients
    2^-4, 2^-3 for the position inputs and the offset / weight projections)."""
    if dtype == torch.float32:
        return nerr(x, ref) <= FP32_LAYER_TOL
    from tests.util import nerr as nerr2
    _, el2 = nerr2(x.double().cpu().numpy(), ref.double().cpu().numpy())
    bound = 2.0 ** -6 if name == "out" else (2.0 ** -3 if any(t in name for t in LOOSE) else 2.0 ** -4)
    return el2 <= bound


def _run_layer(name, dtype, p, patch_dropout=None):
    from tests import module_cases
    gold = np.load(os.path.join(GOLDEN, name + ".npz"))
    case = module_cases.CASES[name]
    module = case["build"]()
    state = {k[len("state."):]: torch.from_numpy(v) for k, v in gold.items() if k.startswith("state.")}
    module.load_state_dict(state, strict=True)
    module = module.to(DEV).to(dtype).train()
    for m in module.modules():
        if type(m) is nn.Dropout:
            m.p = p
    tensors = {}
    for k, v in gold.items():
        if k.startswith("in."):
            t = torch.from_numpy(v).to(DEV)
            if t.is_floating_point() and (t.dtype == torch.float64 or name in module_cases.WIDE):
                t = t.to(dtype)
            if k[3:] in case["wrt"]:
                t = t.requires_grad_(True)
            tensors[k[3:]] = t
    out = case["call"](module, tensors)
    gout = torch.from_numpy(gold["gout"]).to(device=DEV, dtype=out.dtype)
    params = dict(module.named_parameters())
    grads = torch.autograd.grad(out, [tensors[k] for k in case["wrt"]] + list(params.values()), gout, allow_unused=True)
    names = list(case["wrt"]) + list(params)
    return out.detach(), dict(zip(names, grads))


# bf16: the layers whose bf16 bounds the training tests state (the d_model-256 goldens); the decoder and U-DF goldens
# are d_model 128 and are checked in fp32, where the comparison is tight
BF16_LAYERS = ["layer_encoder_c256", "layer_fusion_v2_c256", "layer_late_fusion_c256"]


@pytest.mark.parametrize("name,dtype", [(n, torch.float32) for n in LAYERS] + [(n, torch.bfloat16) for n in BF16_LAYERS])
def test_layers_train_with_dropout_match_masked_composition(keys, monkeypatch, name, dtype):
    p = 0.1
    out, grads = _run_layer(name, dtype, p)
    assert keys, "no dropout site took the package path"
    recorded = list(keys)
    it = iter(recorded)

    def masked_forward(self, x):             # the reference: each nn.Dropout call takes the next recorded mask
        key = next(it)
        return x * oracle_mask(key, x.shape, self.p).to(x.dtype) * rule(self.p)[1]
    monkeypatch.setattr(nn.Dropout, "forward", masked_forward)
    out64, grads64 = _run_layer(name, torch.float64, p)
    assert next(it, None) is None, "the reference used fewer dropout calls than the package path"
    assert _within_layer_bounds(dtype, "out", out, out64)
    for k, g in grads.items():
        if g is None:
            assert grads64[k] is None or float(grads64[k].abs().max()) == 0
            continue
        assert _within_layer_bounds(dtype, k, g, grads64[k]), k


# ---------------------------------------------------------------------------------------------------------------------
# CUDA graphs
def test_graphed_train_step_with_dropout_draws_fresh_masks():
    from dfvod_b200 import data_parallel
    from dfvod_b200 import transformer_layers as tl
    torch.manual_seed(0)
    shapes = [(12, 16), (6, 8)]
    s = sum(h * w for h, w in shapes)
    st = torch.as_tensor(shapes, dtype=torch.long, device=DEV)
    ls = torch.as_tensor([0, 12 * 16], dtype=torch.long, device=DEV)
    enc = tl.DeformableTransformerEncoder(tl.DeformableTransformerEncoderLayer(256, 512, 0.1, "relu", 2, 8, 4), 2)
    enc = enc.to(DEV).bfloat16().train()
    src = torch.randn(2, s, 256, device=DEV).bfloat16()
    pos = torch.randn(2, s, 256, device=DEV).bfloat16()
    vr = torch.ones(2, 2, 2, device=DEV)
    opt = torch.optim.SGD(enc.parameters(), lr=0.0)           # parameters stay put: only the masks change the loss
    step = data_parallel.GraphedTrainStep(enc, opt, lambda: enc(src, st, ls, vr, pos, None).float().square().mean(),
                                          warmup=2)
    losses = [float(step()) for _ in range(3)]
    torch.cuda.synchronize()
    assert all(np.isfinite(losses))
    assert len(set(losses)) == 3, losses
