"""GPU: bf16 training of the linear layers on the package's own kernels (csrc/linear_bf16.cu).

    forward   y  = x W^T + b            linear_bf16
    backward  dx = g W                  linear_bf16 with W^T as its weight
              dW = g^T x, db = sum g    linear_bf16_wgrad: one pass over g, split-K partials summed in a fixed order

Bounds: a kernel against the fp64 product of the same bf16 operands, 2^-8 of the output range (one bf16 rounding of an
fp32-accumulated result, as for the forward kernel); gradients through autograd 2^-7; whole layers the stated bf16 layer
bounds of test_gpu_modules.py against the reference classes in fp64."""
import copy

import pytest
import torch
import torch.nn.functional as F

from dfvod_b200 import _lib
from dfvod_b200.ops.functions import layer_epilogue_func as L
from dfvod_b200.ops.functions import linear, linear_relu, linear_zero_rows

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
INVALID_VALUE = 1          # cudaErrorInvalidValue

SHAPES = [(256, 256), (384, 256), (1024, 256), (256, 1024), (64, 64), (192, 256)]     # (out, in)


def nerr(x, ref):
    return float((x.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-300))


def operands(rows, n, k, seed):
    torch.manual_seed(seed)
    g = (torch.randn(rows, n, device=DEV) / 4).bfloat16()
    x = (torch.randn(rows, k, device=DEV) * 2).bfloat16()
    return g, x


@pytest.mark.parametrize("n,k", SHAPES)
@pytest.mark.parametrize("rows", [1, 127, 129, 5000, 88892])
@pytest.mark.parametrize("with_bias", [True, False])
def test_wgrad_kernel_matches_fp64(rows, n, k, with_bias):
    g, x = operands(rows, n, k, rows + n + k)
    dw, db = L.linear_bf16_wgrad(g, x, with_bias=with_bias)
    torch.cuda.synchronize()
    assert dw.shape == (n, k) and dw.dtype == torch.bfloat16
    assert nerr(dw, g.double().t() @ x.double()) <= 2.0 ** -8
    if with_bias:
        assert db.shape == (n,) and db.dtype == torch.bfloat16
        assert nerr(db, g.double().sum(0)) <= 2.0 ** -8
    else:
        assert db is None


@pytest.mark.parametrize("rows", [1, 129, 5000])
def test_wgrad_kernel_is_deterministic_and_writes_only_its_outputs(rows):
    """Two calls give the same bits; dW and db placed in the middle of sentinel-filled buffers: nothing around them
    changes (C ABI called directly)."""
    lib = _lib.load()
    stream = torch.cuda.current_stream().cuda_stream
    n, k, pad = 192, 320, 64
    g, x = operands(rows, n, k, rows)
    floats = lib.msda_layer_linear_bf16_wgrad_scratch_floats(rows, n, k)
    assert floats > 0
    scratch = torch.empty(floats, device=DEV)
    outs = []
    for _ in range(2):
        big_w = torch.full((pad + n * k + pad,), 7.0, device=DEV, dtype=torch.bfloat16)
        big_b = torch.full((pad + n + pad,), 7.0, device=DEV, dtype=torch.bfloat16)
        dw, db = big_w[pad:pad + n * k], big_b[pad:pad + n]
        _lib.check(lib.msda_layer_linear_bf16_wgrad(g.data_ptr(), x.data_ptr(), rows, n, k, dw.data_ptr(), db.data_ptr(),
                                                    scratch.data_ptr(), floats, stream), "wgrad")
        torch.cuda.synchronize()
        for big in (big_w, big_b):
            assert bool((big[:pad] == 7.0).all()) and bool((big[-pad:] == 7.0).all())
        outs.append((dw.clone(), db.clone()))
        scratch.fill_(float("nan"))                      # the partials are rewritten, never accumulated into
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    assert nerr(outs[0][0].view(n, k), g.double().t() @ x.double()) <= 2.0 ** -8
    assert nerr(outs[0][1], g.double().sum(0)) <= 2.0 ** -8


def test_wgrad_kernel_refuses_what_it_does_not_take():
    lib = _lib.load()
    stream = torch.cuda.current_stream().cuda_stream
    rows, n, k = 300, 128, 256
    g, x = operands(rows, n, k, 0)
    dw = torch.empty(n, k, device=DEV, dtype=torch.bfloat16)
    db = torch.empty(n, device=DEV, dtype=torch.bfloat16)
    floats = lib.msda_layer_linear_bf16_wgrad_scratch_floats(rows, n, k)
    scratch = torch.empty(floats + 8, device=DEV)
    call = lambda rows_, n_, k_, sc_floats, g_ptr=g.data_ptr(), sc=scratch.data_ptr(): lib.msda_layer_linear_bf16_wgrad(
        g_ptr, x.data_ptr(), rows_, n_, k_, dw.data_ptr(), db.data_ptr(), sc, sc_floats, stream)
    # shapes: features / inputs not a multiple of 64, no rows
    for n_, k_ in ((96, 256), (128, 200), (0, 256)):
        assert not lib.msda_layer_linear_bf16_wgrad_supported(n_, k_)
        assert lib.msda_layer_linear_bf16_wgrad_scratch_floats(rows, n_, k_) == 0
        assert call(rows, n_, k_, floats) == INVALID_VALUE
    assert lib.msda_layer_linear_bf16_wgrad_scratch_floats(0, n, k) == 0
    assert call(0, n, k, floats) == INVALID_VALUE
    # scratch one float short, misaligned scratch, misaligned operand
    assert call(rows, n, k, floats - 1) == INVALID_VALUE
    assert call(rows, n, k, floats, sc=scratch.data_ptr() + 4) == INVALID_VALUE
    assert call(rows, n, k, floats, g_ptr=g.data_ptr() + 2) == INVALID_VALUE
    assert call(rows, n, k, floats) == 0
    torch.cuda.synchronize()
    assert nerr(dw, g.double().t() @ x.double()) <= 2.0 ** -8


@pytest.fixture
def spy(monkeypatch):
    """Lowers the training threshold to 1024 rows and counts the kernel calls of the bf16 training route."""
    calls = {"fwd": 0, "wgrad": 0}
    fwd, wgrad = L.linear_bf16, L.linear_bf16_wgrad

    def fwd_spy(*a, **kw):
        calls["fwd"] += 1
        return fwd(*a, **kw)

    def wgrad_spy(*a, **kw):
        calls["wgrad"] += 1
        return wgrad(*a, **kw)

    monkeypatch.setattr(L, "linear_bf16", fwd_spy)
    monkeypatch.setattr(L, "linear_bf16_wgrad", wgrad_spy)
    monkeypatch.setattr(L, "BF16_TRAIN_KERNEL_MIN_ROWS", 1024)
    return calls


def _grads(fn, lin, x, g):
    x = x.detach().clone().requires_grad_(True)
    lin.zero_grad(set_to_none=True)
    y = fn(lin, x)
    y.backward(g)
    return y.detach(), x.grad, lin.weight.grad, lin.bias.grad


@pytest.mark.parametrize("kind", ["linear", "linear_relu", "linear_zero_rows"])
def test_training_route_matches_fp64(spy, kind):
    torch.manual_seed(11)
    rows = 3000
    lin = torch.nn.Linear(256, 384).to(DEV).bfloat16()
    x = torch.randn(rows, 256, device=DEV).bfloat16()
    mask = torch.rand(rows, device=DEV) < 0.2
    fn = {"linear": linear, "linear_relu": linear_relu,
          "linear_zero_rows": lambda m, t: linear_zero_rows(m, t, mask)}[kind]
    g = torch.randn(rows, 384, device=DEV).bfloat16()
    y, dx, dw, db = _grads(fn, lin, x, g)
    # forward + input gradient on linear_bf16, weight + bias gradient in one linear_bf16_wgrad
    assert spy == {"fwd": 2, "wgrad": 1}
    x64, w64 = x.double(), lin.weight.double()
    pre = x64 @ w64.t() + lin.bias.double()
    g64 = g.double()
    if kind == "linear_relu":
        pre = pre.relu()
        g64 = g64 * (y > 0)                              # the mask the backward applies: the kernel's own output
    if kind == "linear_zero_rows":
        pre = pre.masked_fill(mask[:, None], 0.0)
        g64 = g64.masked_fill(mask[:, None], 0.0)
    assert nerr(y, pre) <= 2.0 ** -7
    assert nerr(dx, g64 @ w64) <= 2.0 ** -7
    assert nerr(dw, g64.t() @ x64) <= 2.0 ** -7
    assert nerr(db, g64.sum(0)) <= 2.0 ** -7
    # below the threshold: the library path, bit for bit what it gives without the route
    spy["fwd"] = spy["wgrad"] = 0
    few = _grads(fn if kind != "linear_zero_rows" else (lambda m, t: linear_zero_rows(m, t, mask[:1000])), lin, x[:1000],
                 g[:1000])
    assert spy == {"fwd": 0, "wgrad": 0}
    L.BF16_TRAIN_KERNEL_MIN_ROWS = None
    lib = _grads(fn if kind != "linear_zero_rows" else (lambda m, t: linear_zero_rows(m, t, mask[:1000])), lin, x[:1000],
                 g[:1000])
    assert all(torch.equal(a, b) for a, b in zip(few, lib))


def test_training_route_under_autocast(spy):
    """fp32 parameters under torch.autocast(bfloat16): the GEMMs run in bf16 on the kernels, gradients come back in the
    parameters' dtype."""
    torch.manual_seed(12)
    rows = 2500
    lin = torch.nn.Linear(256, 256).to(DEV)
    x = torch.randn(rows, 256, device=DEV)
    g = torch.randn(rows, 256, device=DEV)
    xr = x.detach().clone().requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        y = linear(lin, xr)
    assert y.dtype == torch.bfloat16
    y.backward(g.bfloat16())
    y = y.detach()
    assert spy == {"fwd": 2, "wgrad": 1}
    assert lin.weight.grad.dtype == torch.float32 and lin.bias.grad.dtype == torch.float32
    xb, wb, bb, gb = (t.bfloat16().double() for t in (x, lin.weight, lin.bias, g))
    assert nerr(y, xb @ wb.t() + bb) <= 2.0 ** -7
    assert nerr(xr.grad, gb @ wb) <= 2.0 ** -7
    assert nerr(lin.weight.grad, gb.t() @ xb) <= 2.0 ** -7
    assert nerr(lin.bias.grad, gb.sum(0)) <= 2.0 ** -7


def test_other_dtypes_and_shapes_keep_the_library(spy):
    """fp32 and fp16 training, and the bf16 shape where the library is faster (256 <- 1024), keep the library GEMMs."""
    torch.manual_seed(13)
    for dtype, k in ((torch.float32, 256), (torch.float16, 256), (torch.bfloat16, 1024)):
        lin = torch.nn.Linear(k, 256).to(DEV).to(dtype)
        x = torch.randn(2048, k, device=DEV).to(dtype).requires_grad_(True)
        linear(lin, x).float().sum().backward()
        linear_relu(lin, x).float().sum().backward()
    assert spy == {"fwd": 0, "wgrad": 0}


LAYERS = ["layer_encoder_c256", "layer_fusion_v2_c256", "layer_fusion_v2_c256_l2", "layer_late_fusion_c256"]


@pytest.mark.parametrize("name", LAYERS)
def test_layers_train_on_the_kernels_within_bf16_bounds(spy, name):
    """Every linear of the layer on the training route (threshold 1): the stated bf16 layer bounds of
    test_gpu_modules.py against the reference class in fp64."""
    from tests import module_cases
    from tests.util import load_golden, nerr as nerr2
    L.BF16_TRAIN_KERNEL_MIN_ROWS = 1
    gold = load_golden(name)
    out, gin, gpar = module_cases.run_case(name, gold, "cuda", torch.bfloat16)
    assert spy["wgrad"] > 0
    loose_in = ("pos", "query_pos")
    emax, el2 = nerr2(out, gold["out"])
    assert emax <= 2.0 ** -5 and el2 <= 2.0 ** -6, f"out: {emax:.2e} {el2:.2e}"
    for k, g in gin.items():
        emax, el2 = nerr2(g, gold["grad_in." + k])
        if k in loose_in:
            assert el2 <= 2.0 ** -3, f"{k}: {emax:.2e} {el2:.2e}"
        else:
            assert emax <= 2.0 ** -3 and el2 <= 2.0 ** -5, f"{k}: {emax:.2e} {el2:.2e}"
    for k, g in gpar.items():
        ref = gold.get("grad_param." + k)
        if ref is None or ref.shape == () or g is None:
            continue
        emax, el2 = nerr2(g, ref)
        loose = "sampling_offsets" in k or "attention_weights" in k
        assert el2 <= (2.0 ** -3 if loose else 2.0 ** -4), f"{k}: {emax:.2e} {el2:.2e}"


def test_graphed_train_step_on_the_kernels_matches_eager(spy):
    """GraphedTrainStep of a bf16 encoder with every linear on the training route: the same losses and parameters as the
    eager steps (the weight-gradient kernel allocates nothing and synchronises nothing, so it is captured as is)."""
    from dfvod_b200 import data_parallel
    from dfvod_b200 import transformer_layers as tl
    L.BF16_TRAIN_KERNEL_MIN_ROWS = 256
    torch.manual_seed(0)
    shapes = [(12, 16), (6, 8)]
    s = sum(h * w for h, w in shapes)
    st = torch.as_tensor(shapes, dtype=torch.long, device=DEV)
    ls = torch.as_tensor([0, 12 * 16], dtype=torch.long, device=DEV)
    enc = tl.DeformableTransformerEncoder(tl.DeformableTransformerEncoderLayer(256, 512, 0.0, "relu", 2, 8, 4), 2).to(DEV)
    with torch.no_grad():
        for p in enc.parameters():
            p.add_(torch.randn_like(p) * 0.02)
    enc = enc.bfloat16()
    enc2 = copy.deepcopy(enc)
    src = torch.randn(2, s, 256, device=DEV).bfloat16()
    pos = torch.randn(2, s, 256, device=DEV).bfloat16()
    vr = torch.ones(2, 2, 2, device=DEV)                 # fp32, as DeformableTransformer passes them
    loss_of = lambda m: m(src, st, ls, vr, pos, None).float().square().mean()

    opt = torch.optim.SGD(enc.parameters(), lr=0.5)
    losses = []
    for _ in range(2):
        opt.zero_grad(set_to_none=True)
        loss = loss_of(enc)
        loss.backward()
        opt.step()
        losses.append(float(loss))
    assert spy["wgrad"] > 0
    opt2 = torch.optim.SGD(enc2.parameters(), lr=0.5)
    step = data_parallel.GraphedTrainStep(enc2, opt2, lambda: loss_of(enc2), warmup=2)
    glosses = [float(step()) for _ in range(2)]
    torch.cuda.synchronize()
    for a, b in zip(losses, glosses):
        assert abs(a - b) <= 1e-3 * abs(a), (losses, glosses)
    for (name, p), q in zip(enc.named_parameters(), enc2.parameters()):
        # bf16 parameters: the deformable-attention backward accumulates with atomics, so the two runs may round a
        # gradient differently and an updated parameter may land on a neighbouring bf16 value
        err = float((p.double() - q.double()).abs().max() / p.double().abs().max().clamp_min(1e-12))
        assert err <= 2.0 ** -6, (name, err)
