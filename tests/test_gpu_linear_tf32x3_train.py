"""GPU: fp32 training of the linear layers on the three-term TF32 kernels (csrc/linear_tf32x3.cu),
set_fp32_train_gemm_mode("tf32x3").

    forward   y  = x W^T + b            linear_tf32x3 with the split (W_hi, W_lo)
    backward  dx = g W                  linear_tf32x3 with (W_hi^T, W_lo^T) as its weight pair
              dW = g^T x, db = sum g    linear_tf32x3_wgrad: both operands split in shared memory, one pass over g,
                                        split-K partials summed in a fixed order

Bounds: BASELINE's fp32 bound, 1e-5 of the output range against fp64, and for the weight-gradient kernel also at most twice
the error of the IEEE SGEMM on the same operands (+ 1e-7 absolute for sums that cancel to almost nothing)."""
import copy

import pytest
import torch

from dfvod_b200 import _lib
from dfvod_b200.ops.functions import layer_epilogue_func as L
from dfvod_b200.ops.functions import linear, linear_relu, linear_zero_rows, set_fp32_train_gemm_mode

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
INVALID_VALUE = 1          # cudaErrorInvalidValue

SHAPES = [(256, 256), (384, 256), (1024, 256), (256, 1024), (64, 64), (192, 256), (32, 64), (96, 256)]   # (out, in)


def nerr(x, ref):
    return float((x.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-300))


def abs_err(x, ref):
    return float((x.double() - ref).abs().max())


def operands(rows, n, k, seed):
    torch.manual_seed(seed)
    return torch.randn(rows, n, device=DEV) / 4, torch.randn(rows, k, device=DEV) * 2


@pytest.fixture
def ieee():
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32 = prev


@pytest.mark.parametrize("n,k", SHAPES)
@pytest.mark.parametrize("rows", [1, 127, 129, 5000, 88892])
@pytest.mark.parametrize("with_bias", [True, False])
def test_wgrad_kernel_matches_fp64(ieee, rows, n, k, with_bias):
    g, x = operands(rows, n, k, rows + n + k)
    dw, db = L.linear_tf32x3_wgrad(g, x, with_bias=with_bias)
    torch.cuda.synchronize()
    assert dw.shape == (n, k) and dw.dtype == torch.float32
    ref_w = g.double().t() @ x.double()
    sgemm_w = g.t() @ x
    assert nerr(dw, ref_w) <= 1e-5
    if rows > 1:
        assert abs_err(dw, ref_w) <= 2 * abs_err(sgemm_w, ref_w) + 1e-7
    else:
        # one row is one product per output and no sum: the SGEMM's only error is the rounding of that product (2^-24
        # of it), while the split drops g_lo x_lo (< 2^-20 of the product) and rounds g_lo / x_lo to TF32 (< 2^-21 each):
        # measured 4-8x the SGEMM's error here.  The split's own bound, element by element:
        assert bool(((dw.double() - ref_w).abs() <= 2.0 ** -19 * ref_w.abs()).all())
    if with_bias:
        assert db.shape == (n,) and db.dtype == torch.float32
        ref_b = g.double().sum(0)
        assert nerr(db, ref_b) <= 1e-5
        assert abs_err(db, ref_b) <= 2 * abs_err(g.sum(0), ref_b) + 1e-7
    else:
        assert db is None


@pytest.mark.parametrize("rows", [1, 129, 5000])
def test_wgrad_kernel_is_deterministic_and_writes_only_its_outputs(rows):
    """Two calls give the same bits; dW and db placed in the middle of sentinel-filled buffers: nothing around them
    changes (C ABI called directly)."""
    lib = _lib.load()
    stream = torch.cuda.current_stream().cuda_stream
    n, k, pad = 160, 352, 64
    g, x = operands(rows, n, k, rows)
    floats = lib.msda_layer_linear_tf32x3_wgrad_scratch_floats(rows, n, k)
    assert floats > 0
    scratch = torch.empty(floats, device=DEV)
    outs = []
    for _ in range(2):
        big_w = torch.full((pad + n * k + pad,), 7.0, device=DEV)
        big_b = torch.full((pad + n + pad,), 7.0, device=DEV)
        dw, db = big_w[pad:pad + n * k], big_b[pad:pad + n]
        _lib.check(lib.msda_layer_linear_tf32x3_wgrad(g.data_ptr(), x.data_ptr(), rows, n, k, dw.data_ptr(),
                                                      db.data_ptr(), scratch.data_ptr(), floats, stream), "wgrad")
        torch.cuda.synchronize()
        for big in (big_w, big_b):
            assert bool((big[:pad] == 7.0).all()) and bool((big[-pad:] == 7.0).all())
        outs.append((dw.clone(), db.clone()))
        scratch.fill_(float("nan"))                      # the partials are rewritten, never accumulated into
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    assert nerr(outs[0][0].view(n, k), g.double().t() @ x.double()) <= 1e-5
    assert nerr(outs[0][1], g.double().sum(0)) <= 1e-5


def test_wgrad_kernel_refuses_what_it_does_not_take():
    lib = _lib.load()
    stream = torch.cuda.current_stream().cuda_stream
    rows, n, k = 300, 128, 256
    g, x = operands(rows, n, k, 0)
    dw = torch.empty(n, k, device=DEV)
    db = torch.empty(n, device=DEV)
    floats = lib.msda_layer_linear_tf32x3_wgrad_scratch_floats(rows, n, k)
    scratch = torch.empty(floats + 8, device=DEV)
    call = lambda rows_, n_, k_, sc_floats, g_ptr=g.data_ptr(), sc=scratch.data_ptr(): lib.msda_layer_linear_tf32x3_wgrad(
        g_ptr, x.data_ptr(), rows_, n_, k_, dw.data_ptr(), db.data_ptr(), sc, sc_floats, stream)
    # shapes: features / inputs not a multiple of 32, none, negative
    for n_, k_ in ((48, 256), (128, 200), (0, 256), (128, 0), (-32, 64)):
        assert not lib.msda_layer_linear_tf32x3_wgrad_supported(n_, k_)
        assert lib.msda_layer_linear_tf32x3_wgrad_scratch_floats(rows, n_, k_) == 0
        assert call(rows, n_, k_, floats) == INVALID_VALUE
    assert lib.msda_layer_linear_tf32x3_wgrad_scratch_floats(0, n, k) == 0
    assert call(0, n, k, floats) == INVALID_VALUE
    # scratch one float short, misaligned scratch, misaligned operand
    assert call(rows, n, k, floats - 1) == INVALID_VALUE
    assert call(rows, n, k, floats, sc=scratch.data_ptr() + 4) == INVALID_VALUE
    assert call(rows, n, k, floats, g_ptr=g.data_ptr() + 4) == INVALID_VALUE
    assert call(rows, n, k, floats) == 0
    torch.cuda.synchronize()
    assert nerr(dw, g.double().t() @ x.double()) <= 1e-5


@pytest.fixture
def spy(monkeypatch):
    """Mode "tf32x3", the training threshold lowered to 1024 rows, and the kernel calls of the fp32 training route
    counted (forward and dx: _linear_tf32x3_kernel; dW + db: linear_tf32x3_wgrad).  The mode is restored afterwards."""
    calls = {"fwd": 0, "wgrad": 0}
    fwd, wgrad = L._linear_tf32x3_kernel, L.linear_tf32x3_wgrad

    def fwd_spy(*a, **kw):
        calls["fwd"] += 1
        return fwd(*a, **kw)

    def wgrad_spy(*a, **kw):
        calls["wgrad"] += 1
        return wgrad(*a, **kw)

    monkeypatch.setattr(L, "_linear_tf32x3_kernel", fwd_spy)
    monkeypatch.setattr(L, "linear_tf32x3_wgrad", wgrad_spy)
    monkeypatch.setattr(L, "FP32_TRAIN_KERNEL_MIN_ROWS", 1024)
    prev = set_fp32_train_gemm_mode("tf32x3")
    yield calls
    set_fp32_train_gemm_mode(prev)


def _grads(fn, lin, x, g):
    x = x.detach().clone().requires_grad_(True)
    lin.zero_grad(set_to_none=True)
    y = fn(lin, x)
    y.backward(g)
    return y.detach(), x.grad, lin.weight.grad, lin.bias.grad


@pytest.mark.parametrize("kind", ["linear", "linear_relu", "linear_zero_rows"])
def test_training_route_matches_fp64(ieee, spy, kind):
    torch.manual_seed(11)
    rows = 3000
    lin = torch.nn.Linear(256, 384).to(DEV)
    x = torch.randn(rows, 256, device=DEV)
    mask = torch.rand(rows, device=DEV) < 0.2
    fn = {"linear": linear, "linear_relu": linear_relu,
          "linear_zero_rows": lambda m, t: linear_zero_rows(m, t, mask)}[kind]
    g = torch.randn(rows, 384, device=DEV)
    y, dx, dw, db = _grads(fn, lin, x, g)
    # forward + input gradient on linear_tf32x3, weight + bias gradient in one linear_tf32x3_wgrad
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
    assert nerr(y, pre) <= 1e-5
    assert nerr(dx, g64 @ w64) <= 1e-5
    assert nerr(dw, g64.t() @ x64) <= 1e-5
    assert nerr(db, g64.sum(0)) <= 1e-5
    few_fn = fn if kind != "linear_zero_rows" else (lambda m, t: linear_zero_rows(m, t, mask[:1000]))
    # below the threshold, and in the default mode: the library path, bit for bit what it gives without the route
    spy["fwd"] = spy["wgrad"] = 0
    few = _grads(few_fn, lin, x[:1000], g[:1000])
    set_fp32_train_gemm_mode("library")
    full = _grads(fn, lin, x, g)
    assert spy == {"fwd": 0, "wgrad": 0}
    L.FP32_TRAIN_KERNEL_MIN_ROWS = None
    set_fp32_train_gemm_mode("tf32x3")
    lib_few = _grads(few_fn, lin, x[:1000], g[:1000])
    lib_full = _grads(fn, lin, x, g)
    assert spy == {"fwd": 0, "wgrad": 0}
    assert all(torch.equal(a, b) for a, b in zip(few, lib_few))
    assert all(torch.equal(a, b) for a, b in zip(full, lib_full))


def test_autocast_and_16_bit_inputs_never_take_the_route(spy):
    """fp32 parameters under torch.autocast, and bf16 / fp16 layers: the fp32 training route is not taken."""
    torch.manual_seed(13)
    lin = torch.nn.Linear(256, 256).to(DEV)
    x = torch.randn(2048, 256, device=DEV).requires_grad_(True)
    for adt in (torch.bfloat16, torch.float16):
        with torch.autocast("cuda", dtype=adt):
            y1, y2 = linear(lin, x), linear_relu(lin, x)
        (y1.float().sum() + y2.float().sum()).backward()
    for dtype in (torch.bfloat16, torch.float16):
        lin16 = copy.deepcopy(lin).to(dtype)
        x16 = x.detach().to(dtype).requires_grad_(True)
        linear(lin16, x16).float().sum().backward()
        linear_relu(lin16, x16).float().sum().backward()
    assert spy == {"fwd": 0, "wgrad": 0}


def test_set_fp32_train_gemm_mode():
    assert L.FP32_TRAIN_GEMM_MODE == "library"               # the default: the reference's own arithmetic
    assert set_fp32_train_gemm_mode("tf32x3") == "library"
    try:
        assert set_fp32_train_gemm_mode("tf32x3") == "tf32x3"
        with pytest.raises(ValueError):
            set_fp32_train_gemm_mode("fp8")
        assert L.FP32_TRAIN_GEMM_MODE == "tf32x3"
    finally:
        assert set_fp32_train_gemm_mode("library") == "tf32x3"


def _routable(module):
    """Whether a module has an nn.Linear with bias whose shape the route takes (the linears of the package go through
    linear / linear_relu / linear_zero_rows)."""
    lib = _lib.load()
    return any(isinstance(m, torch.nn.Linear) and m.bias is not None
               and L._fp32_train_kernels_win(m.out_features, m.in_features)
               and lib.msda_layer_linear_tf32x3_wgrad_supported(m.out_features, m.in_features)
               and lib.msda_layer_linear_tf32x3_supported(m.in_features, m.out_features)
               for m in module.modules())


def _module_cases():
    from tests import module_cases
    return sorted(module_cases.CASES)


@pytest.mark.parametrize("name", _module_cases())
def test_fp32_layers_train_on_the_kernels_within_fp32_bound(ieee, spy, name):
    """Every linear of the module on the fp32 training route (threshold 1): the 1e-5 bound of
    test_fp32_matches_reference_class (normalised max and relative L2 against the reference class in fp64) for the
    output and every gradient."""
    from tests import module_cases
    from tests.util import load_golden, nerr as nerr2
    L.FP32_TRAIN_KERNEL_MIN_ROWS = 1
    gold = load_golden(name)
    out, gin, gpar = module_cases.run_case(name, gold, "cuda", torch.float32)
    if _routable(module_cases.CASES[name]["build"]()):
        assert spy["wgrad"] > 0
    emax, el2 = nerr2(out, gold["out"])
    assert emax <= 1e-5 and el2 <= 1e-5, f"out: {emax:.2e} {el2:.2e}"
    for k, g in gin.items():
        if gold["grad_in." + k].shape == () or g is None:
            continue
        emax, el2 = nerr2(g, gold["grad_in." + k])
        assert emax <= 1e-5 and el2 <= 1e-5, f"{k}: {emax:.2e} {el2:.2e}"
    for k, g in gpar.items():
        ref = gold.get("grad_param." + k)
        if ref is None or ref.shape == () or g is None:
            continue
        emax, el2 = nerr2(g, ref)
        assert emax <= 1e-5 and el2 <= 1e-5, f"{k}: {emax:.2e} {el2:.2e}"


def test_graphed_train_step_on_the_kernels_matches_eager(ieee, spy):
    """GraphedTrainStep of an fp32 d_model-256 encoder with every linear on the fp32 training route: the losses and
    parameters of the eager steps (the weight-gradient kernel allocates nothing and synchronises nothing, and the weight
    split is not cached under capture)."""
    from dfvod_b200 import data_parallel
    from dfvod_b200 import transformer_layers as tl
    L.FP32_TRAIN_KERNEL_MIN_ROWS = 256
    torch.manual_seed(0)
    shapes = [(12, 16), (6, 8)]
    s = sum(h * w for h, w in shapes)
    st = torch.as_tensor(shapes, dtype=torch.long, device=DEV)
    ls = torch.as_tensor([0, 12 * 16], dtype=torch.long, device=DEV)
    enc = tl.DeformableTransformerEncoder(tl.DeformableTransformerEncoderLayer(256, 512, 0.0, "relu", 2, 8, 4), 2).to(DEV)
    with torch.no_grad():
        for p in enc.parameters():
            p.add_(torch.randn_like(p) * 0.02)
    enc2 = copy.deepcopy(enc)
    src = torch.randn(2, s, 256, device=DEV)
    pos = torch.randn(2, s, 256, device=DEV)
    vr = torch.ones(2, 2, 2, device=DEV)
    loss_of = lambda m: m(src, st, ls, vr, pos, None).square().mean()

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
        assert abs(a - b) <= 1e-5 * abs(a), (losses, glosses)
    for (name, p), q in zip(enc.named_parameters(), enc2.parameters()):
        # the deformable-attention backward accumulates with atomics: last-bit differences in a gradient
        err = float((p.double() - q.double()).abs().max() / p.double().abs().max().clamp_min(1e-12))
        assert err <= 1e-5, (name, err)
