"""GPU: the deterministic backward (C ABI msda_backward_deterministic, msda_fused_backward_deterministic,
msda_roi_align_backward_deterministic; DESIGN.md section 3.15), taken whenever torch.use_deterministic_algorithms is
on.  Bitwise repeatability, independence of the query / RoI order, parity with the fp64 oracles at the tolerances of the
existing parity tests, edge cases, write bounds, CUDA-graph capture and bitwise reproducible training."""
import contextlib
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch

from tests import util
from oracle import c_oracle, roi_align_oracle

from dfvod_b200 import _lib
from dfvod_b200 import MultiScaleDeformableAttention as MSDA
from dfvod_b200 import MSDeformAttnFunction
from dfvod_b200.ops.functions import MSDeformAttnFusedFunction
from dfvod_b200.temporal_stage import roi_align_tokens

pytestmark = pytest.mark.gpu
DEV = "cuda"
INVALID_VALUE = 1                                    # cudaErrorInvalidValue
TOL = {torch.float32: (1e-5, 1e-5), torch.bfloat16: (2.0 ** -7, 4e-3), torch.float64: (1e-9, 1e-9)}
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@contextlib.contextmanager
def deterministic(on=True, warn_only=False):
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(on, warn_only=warn_only)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_warn)


def bits_equal(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.uint8), b.contiguous().view(torch.uint8))


# ------------------------------------------------------------------ the plain op
PLAIN = [
    # shapes, N, M, D, Lq, P
    ([(20, 30), (10, 15), (5, 8), (3, 4)], 2, 8, 32, 257, 4),       # fast kernel
    ([(6, 6), (3, 3)], 2, 3, 30, 40, 2),                            # D = 30: generic kernel
]
PLAIN_IDS = ["D32", "D30"]


def plain_inputs(case, dtype, seed=5):
    shapes, n, m, d, lq, p = case
    value, loc, attn, gout = util.make_inputs(shapes, n, m, d, lq, p, seed=seed, loc_range=(-0.1, 1.1))
    side = torch.float64 if dtype == torch.float64 else torch.float32
    return value.to(dtype), loc.to(side), attn.to(side), gout.reshape(n, lq, m * d).to(dtype)


def plain_backward(shapes, value, loc, attn, gout):
    st, ls = util.shapes_tensors(shapes, DEV)
    gv, gl, ga = MSDA.ms_deform_attn_backward(value.to(DEV), st, ls, loc.to(DEV), attn.to(DEV), gout.to(DEV), 64)
    torch.cuda.synchronize()
    return gv, gl, ga


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float64])
@pytest.mark.parametrize("case", PLAIN, ids=PLAIN_IDS)
def test_plain_repeatable_order_independent_and_exact(case, dtype):
    shapes, n, m, d, lq, p = case
    value, loc, attn, gout = plain_inputs(case, dtype)
    with deterministic():
        first = plain_backward(shapes, value, loc, attn, gout)
        again = plain_backward(shapes, value, loc, attn, gout)
        perm = torch.randperm(lq, generator=torch.Generator().manual_seed(1))
        permuted = plain_backward(shapes, value, loc[:, perm], attn[:, perm], gout[:, perm])
    for x, y in zip(first, again):
        assert bits_equal(x, y)
    assert bits_equal(first[0], permuted[0]), "grad_value depends on the order of the queries"
    assert bits_equal(first[1][:, perm], permuted[1]) and bits_equal(first[2][:, perm], permuted[2])
    args = (value.double().numpy(), shapes, util.lsi_of(shapes), loc.double().numpy(), attn.double().numpy())
    ref = c_oracle.backward(*args, gout.double().numpy())
    max_tol, l2_tol = TOL[dtype]
    for name, x, r in zip(("grad_value", "grad_loc", "grad_attn"), first, ref):
        emax, el2 = util.nerr(x.double().cpu().numpy().reshape(r.shape), r)
        assert emax <= max_tol and el2 <= l2_tol, f"{name}: max {emax:.3e} l2 {el2:.3e}"


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_plain_coco_grid_repeatable_and_order_independent(dtype):
    """Encoder geometry at COCO scale: 22 223 queries on the pixel grid, so many queries hit the same pixels."""
    shapes = util.COCO_SHAPES
    s = sum(h * w for h, w in shapes)
    value, loc, attn, gout = util.make_inputs(shapes, 1, 8, 32, s, 4, seed=3, dist="grid")
    value, gout = value.to(dtype), gout.reshape(1, s, 256).to(dtype)
    perm = torch.randperm(s, generator=torch.Generator().manual_seed(2))
    with deterministic():
        a = plain_backward(shapes, value, loc, attn, gout)
        b = plain_backward(shapes, value, loc, attn, gout)
        c = plain_backward(shapes, value, loc[:, perm], attn[:, perm], gout[:, perm])
    assert bits_equal(a[0], b[0]) and bits_equal(a[0], c[0])
    default = plain_backward(shapes, value, loc, attn, gout)
    max_tol, _ = TOL[dtype]
    assert float((a[0].double() - default[0].double()).abs().max() / default[0].double().abs().max()) <= max_tol


def test_plain_gradcheck_fp64():
    """models/ops/test.py:63-78 (the reference's gradcheck), with the deterministic backward."""
    shapes = [(6, 4), (3, 2)]
    value, loc, attn, _ = util.make_inputs(shapes, 1, 2, 2, 2, 2, seed=0)
    st, ls = util.shapes_tensors(shapes, DEV)
    value, loc, attn = (t.double().to(DEV).requires_grad_(True) for t in (value, loc, attn))
    with deterministic():
        assert torch.autograd.gradcheck(MSDeformAttnFunction.apply, (value, st, ls, loc, attn, 2))


def test_plain_zero_and_nonfinite_grad_output():
    case = PLAIN[0]
    shapes = case[0]
    value, loc, attn, gout = plain_inputs(case, torch.float32)
    with deterministic(warn_only=True):             # warn_only selects the deterministic kernels as well
        gv, gl, ga = plain_backward(shapes, value, loc, attn, torch.zeros_like(gout))
        assert not bool(gv.any()) and not bool(gl.any()) and not bool(ga.any())
        bad = gout.clone()
        bad[0, 3, 5] = float("inf")
        gv, _, _ = plain_backward(shapes, value, loc, attn, bad)
        assert bool(gv.isnan().all()), "a non-finite bound must make all of grad_value NaN"
        bad_attn = attn.clone()
        bad_attn[1, 7, 2, 0, 1] = float("nan")
        gv, _, _ = plain_backward(shapes, value, loc, bad_attn, gout)
        assert bool(gv.isnan().all())


def test_plain_c_abi_refusals_and_write_bounds():
    """MSDA_FLAG_TC and a short scratch are refused; grad_value, grad_loc, grad_attn and the scratch sit between
    sentinel bytes, which stay untouched."""
    lib = _lib.load()
    case = PLAIN[0]
    shapes, n, m, d, lq, p = case
    nl = len(shapes)
    value, loc, attn, gout = (t.to(DEV) for t in plain_inputs(case, torch.bfloat16))
    st, ls = util.shapes_tensors(shapes, DEV)
    stream = torch.cuda.current_stream().cuda_stream
    need = lib.msda_deterministic_scratch_bytes(value.numel(), 0, 0)
    assert need >= value.numel() * 8
    assert lib.msda_deterministic_scratch_bytes(-1, 0, 0) == -1
    pad = 4096
    results = []
    for _ in range(2):
        bufs = {}
        for name, count, dtype in (("gv", value.numel(), torch.bfloat16), ("gl", loc.numel(), torch.float32),
                                   ("ga", attn.numel(), torch.float32), ("scratch", need, torch.uint8)):
            big = torch.full((2 * pad + count,), 7, dtype=dtype, device=DEV)
            bufs[name] = (big, big[pad:pad + count])

        def call(flags, scratch_bytes):
            return lib.msda_backward_deterministic(
                _lib.DTYPE_BF16, gout.data_ptr(), value.data_ptr(), st.data_ptr(), ls.data_ptr(), loc.data_ptr(),
                attn.data_ptr(), n, value.size(1), m, d, nl, lq, p, bufs["gv"][1].data_ptr(), bufs["gl"][1].data_ptr(),
                bufs["ga"][1].data_ptr(), None, flags, bufs["scratch"][1].data_ptr(), scratch_bytes, stream)

        assert call(_lib.FLAG_TC, need) == INVALID_VALUE
        assert call(0, need - 1) == INVALID_VALUE
        _lib.check(call(0, need), "msda_backward_deterministic")
        torch.cuda.synchronize()
        for big, _ in bufs.values():
            assert bool((big[:pad] == 7).all()) and bool((big[-pad:] == 7).all())
        results.append(bufs["gv"][1].clone())
    assert bits_equal(results[0], results[1])


def test_plain_graph_capture_replays_eager_bits():
    case = PLAIN[0]
    shapes = case[0]
    value, loc, attn, gout = (t.to(DEV) for t in plain_inputs(case, torch.float32))
    st, ls = util.shapes_tensors(shapes, DEV)
    with deterministic():
        eager = MSDA.ms_deform_attn_backward(value, st, ls, loc, attn, gout, 64)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            MSDA.ms_deform_attn_backward(value, st, ls, loc, attn, gout, 64)
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            captured = MSDA.ms_deform_attn_backward(value, st, ls, loc, attn, gout, 64)
        for _ in range(2):
            graph.replay()
        torch.cuda.synchronize()
    for x, y in zip(eager, captured):
        assert bits_equal(x, y)


# ------------------------------------------------------------------ the fused op
FUSED = [
    # shapes, N, M, D, Lq, P, ref_dim
    ([(20, 30), (10, 15), (5, 8), (3, 4)], 2, 8, 32, 131, 4, 2),
    ([(20, 30), (10, 15), (5, 8), (3, 4)], 1, 8, 32, 50, 4, 4),
    ([(12, 9), (6, 5)], 2, 4, 16, 39, 3, 2),
]
FUSED_IDS = ["D32_ref2", "D32_ref4", "D16_P3"]


def fused_case(case, seed=7):
    shapes, n, m, d, lq, p, ref_dim = case
    g = torch.Generator().manual_seed(seed)
    nl = len(shapes)
    s = sum(h * w for h, w in shapes)
    value = torch.randn(n, s, m, d, generator=g)
    raw = torch.randn(n, lq, 3 * m * nl * p, generator=g)
    raw[..., :2 * m * nl * p] *= 2.0
    ref = torch.rand(n, lq, nl, 2, generator=g)
    if ref_dim == 4:
        ref = torch.cat([ref, torch.rand(n, lq, nl, 2, generator=g) * 0.5 + 0.05], -1)
    gout = torch.randn(n, lq, m * d, generator=g)
    return value, raw, ref, gout


def fused_backward(shapes, p, value, raw, ref, gout, dtype, ref_grad=True):
    st, ls = util.shapes_tensors(shapes, DEV)
    v = value.to(DEV, dtype).requires_grad_(True)
    # 16-bit raw offsets are read in pairs of points: an odd point count takes fp32 raw (msda_fused_supported)
    rdtype = torch.float32 if p % 2 else dtype
    r = raw.to(DEV, rdtype).requires_grad_(True)
    rf = ref.to(DEV).requires_grad_(ref_grad)
    MSDeformAttnFusedFunction.apply(v, st, ls, rf, r, p).backward(gout.to(DEV, dtype))
    torch.cuda.synchronize()
    return v.grad, r.grad, rf.grad


def fused_oracle(shapes, m, p, value, raw, ref, gout):
    from oracle import msda_oracle
    n, lq = raw.shape[:2]
    nl = len(shapes)
    mlp = m * nl * p
    v, r, rf = (t.double().requires_grad_(True) for t in (value, raw, ref))
    offsets = r[..., :2 * mlp].reshape(n, lq, m, nl, p, 2)
    attn = torch.softmax(r[..., 2 * mlp:].reshape(n, lq, m, nl * p), -1).view(n, lq, m, nl, p)
    if rf.shape[-1] == 2:
        norm = torch.tensor([[w, h] for h, w in shapes], dtype=torch.float64)
        loc = rf[:, :, None, :, None, :] + offsets / norm[None, None, None, :, None, :]
    else:
        loc = rf[:, :, None, :, None, :2] + offsets / p * rf[:, :, None, :, None, 2:] * 0.5
    msda_oracle.core_pytorch(v, shapes, loc, attn).backward(gout.double())
    return v.grad, r.grad, rf.grad


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("case", FUSED, ids=FUSED_IDS)
def test_fused_repeatable_order_independent_and_exact(case, dtype):
    shapes, n, m, d, lq, p, ref_dim = case
    value, raw, ref, gout = fused_case(case)
    if dtype == torch.bfloat16:
        value, raw, gout = (t.bfloat16().float() for t in (value, raw, gout))
    perm = torch.randperm(lq, generator=torch.Generator().manual_seed(4))
    with deterministic():
        a = fused_backward(shapes, p, value, raw, ref, gout, dtype)
        b = fused_backward(shapes, p, value, raw, ref, gout, dtype)
        c = fused_backward(shapes, p, value, raw[:, perm], ref[:, perm], gout[:, perm], dtype)
        no_ref = fused_backward(shapes, p, value, raw, ref, gout, dtype, ref_grad=False)
    for x, y in zip(a, b):
        assert bits_equal(x, y)
    assert bits_equal(a[0], c[0]), "grad_value depends on the order of the queries"
    assert bits_equal(a[1][:, perm], c[1]) and bits_equal(a[2][:, perm], c[2])
    assert no_ref[2] is None and bits_equal(a[0], no_ref[0]) and bits_equal(a[1], no_ref[1])
    if dtype == torch.float32:
        want = fused_oracle(shapes, m, p, value, raw, ref, gout)
        for name, x, w in zip(("grad_value", "grad_raw", "grad_ref"), a, want):
            emax, el2 = util.nerr(x.double().cpu().numpy(), w.numpy())
            assert emax <= 1e-5 and el2 <= 1e-5, f"{name}: max {emax:.3e} l2 {el2:.3e}"
    else:
        default = fused_backward(shapes, p, value, raw, ref, gout, dtype)
        for name, x, w in zip(("grad_value", "grad_raw"), a, default):
            emax, el2 = util.nerr(x.double().cpu().numpy(), w.double().cpu().numpy())
            assert emax <= 2.0 ** -7 and el2 <= 4e-3, f"{name}: max {emax:.3e} l2 {el2:.3e}"


def test_fused_nonfinite_and_write_bounds():
    lib = _lib.load()
    case = FUSED[1]
    shapes, n, m, d, lq, p, ref_dim = case
    nl = len(shapes)
    mlp = m * nl * p
    value, raw, ref, gout = (t.to(DEV) for t in fused_case(case))
    st, ls = util.shapes_tensors(shapes, DEV)
    stream = torch.cuda.current_stream().cuda_stream
    need = lib.msda_deterministic_scratch_bytes(value.numel(), ref.numel(), m)
    assert need >= value.numel() * 8 + ref.numel() * m * 4
    pad = 4096
    bufs = {}
    for name, count, dtype in (("gv", value.numel(), torch.float32), ("graw", raw.numel(), torch.float32),
                               ("gref", ref.numel(), torch.float32), ("scratch", need, torch.uint8)):
        big = torch.full((2 * pad + count,), 7, dtype=dtype, device=DEV)
        bufs[name] = (big, big[pad:pad + count])

    def call(g, scratch_bytes):
        graw = bufs["graw"][1].data_ptr()
        return lib.msda_fused_backward_deterministic(
            _lib.DTYPE_F32, _lib.DTYPE_F32, g.data_ptr(), value.data_ptr(), st.data_ptr(), ls.data_ptr(), ref.data_ptr(),
            ref_dim, raw.data_ptr(), 3 * mlp, raw.data_ptr() + 8 * mlp, 3 * mlp, n, value.size(1), m, d, nl, lq, p,
            bufs["gv"][1].data_ptr(), graw, graw + 8 * mlp, bufs["gref"][1].data_ptr(), None,
            bufs["scratch"][1].data_ptr(), scratch_bytes, stream)

    assert call(gout, need - 1) == INVALID_VALUE
    _lib.check(call(gout, need), "msda_fused_backward_deterministic")
    torch.cuda.synchronize()
    for big, _ in bufs.values():
        assert bool((big[:pad] == 7).all()) and bool((big[-pad:] == 7).all())
    bad = gout.clone()
    bad[0, 1, 2] = float("nan")
    _lib.check(call(bad, need), "msda_fused_backward_deterministic")
    torch.cuda.synchronize()
    assert bool(bufs["gv"][1].isnan().all())
    _lib.check(call(torch.zeros_like(gout), need), "msda_fused_backward_deterministic")
    torch.cuda.synchronize()
    assert not bool(bufs["gv"][1].any()) and not bool(bufs["gref"][1].any())


# ------------------------------------------------------------------ RoIAlign
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float64])
@pytest.mark.parametrize("channels", [256, 30])
def test_roi_align_repeatable_order_independent_and_exact(dtype, channels):
    from tests.test_gpu_roi_align import make_rois
    n, height, width, scale, k = 3, 9, 13, 1 / 32, 40
    g = torch.Generator().manual_seed(channels)
    tokens = torch.randn(n, height * width, channels, generator=g).to(dtype)
    rois = make_rois(n, k, height, width, scale, 7)
    gout = torch.randn(k, 49, channels, generator=g).to(dtype)
    perm = torch.randperm(k, generator=torch.Generator().manual_seed(5))

    def grad(r, go):
        td = tokens.to(DEV).requires_grad_(True)
        roi_align_tokens(td, r.to(DEV), height, width, 7, scale, 2, True).backward(go.to(DEV))
        torch.cuda.synchronize()
        return td.grad

    with deterministic():
        a, b, c = grad(rois, gout), grad(rois, gout), grad(rois[perm], gout[perm])
    assert a.dtype == dtype and bits_equal(a, b) and bits_equal(a, c)
    t64 = tokens.double().clone().requires_grad_(True)
    ref = roi_align_oracle.roi_align_tokens(t64, rois, height, width, 7, scale, 2, True)
    (ref_grad,) = torch.autograd.grad(ref, t64, gout.double())
    tol = {torch.float64: 1e-12, torch.float32: 1e-5, torch.bfloat16: 2.0 ** -7}[dtype]
    assert float((a.double().cpu() - ref_grad).abs().max() / ref_grad.abs().max()) <= tol


def test_roi_align_nonfinite_and_write_bounds():
    from tests.test_gpu_roi_align import make_rois
    lib = _lib.load()
    n, height, width, channels, k = 2, 9, 13, 64, 12
    rois = make_rois(n, k, height, width, 1 / 32, 3).float().to(DEV)
    gout = torch.randn(k, 49, channels, device=DEV)
    count = n * height * width * channels
    need = lib.msda_deterministic_scratch_bytes(count, 0, 0)
    pad = 4096
    big_g = torch.full((2 * pad + count,), 7.0, device=DEV)
    big_s = torch.full((2 * pad + need,), 7, dtype=torch.uint8, device=DEV)
    stream = torch.cuda.current_stream().cuda_stream

    def call(go):
        return lib.msda_roi_align_backward_deterministic(
            _lib.DTYPE_F32, go.data_ptr(), rois.data_ptr(), n, height, width, channels, k, 7, 7, 1 / 32, 2, 1,
            big_g[pad:pad + count].data_ptr(), big_s[pad:pad + need].data_ptr(), need, stream)

    _lib.check(call(gout), "msda_roi_align_backward_deterministic")
    torch.cuda.synchronize()
    for big in (big_g, big_s):
        assert bool((big[:pad] == 7).all()) and bool((big[-pad:] == 7).all())
    bad = gout.clone()
    bad[3, 4, 5] = float("-inf")
    _lib.check(call(bad), "msda_roi_align_backward_deterministic")
    torch.cuda.synchronize()
    assert bool(big_g[pad:pad + count].isnan().all())


# ------------------------------------------------------------------ the flag off changes nothing
def test_flag_off_takes_the_default_symbols(monkeypatch):
    """With the flag off the backward calls msda_backward exactly as before and matches the golden vectors."""
    assert not torch.are_deterministic_algorithms_enabled()
    lib = _lib.load()
    called = []

    class Spy:
        def __getattr__(self, name):
            called.append(name)
            return getattr(lib, name)

    monkeypatch.setattr(_lib, "_lib", Spy())
    g = util.load_golden("op_d32_l4")
    t = {k: torch.from_numpy(v) for k, v in g.items()}
    shapes = [tuple(x) for x in g["shapes"].tolist()]
    gv, gl, ga = plain_backward(shapes, t["value"], t["loc"], t["attn"], t["grad_out"])
    assert "msda_backward" in called and not any(c.endswith("_deterministic") for c in called)
    args = (t["value"].double().numpy(), shapes, util.lsi_of(shapes), t["loc"].double().numpy(),
            t["attn"].double().numpy())
    ref = c_oracle.backward(*args, t["grad_out"].double().numpy())
    tol = 1e-9 if g["value"].dtype == np.float64 else 1e-5
    for x, r in zip((gv, gl, ga), ref):
        emax, _ = util.nerr(x.double().cpu().numpy().reshape(r.shape), r)
        assert emax <= tol


# ------------------------------------------------------------------ training, end to end
TRAIN = textwrap.dedent("""
    import hashlib, sys
    import torch
    torch.use_deterministic_algorithms(True)
    from dfvod_b200.deformable_transformer import DeformableTransformer, _flatten_levels, _shape_tensors
    from dfvod_b200.ops.functions import set_fp32_train_gemm_mode
    dtype = {"bf16": torch.bfloat16, "fp32": torch.float32}[sys.argv[1]]
    if dtype == torch.float32:
        set_fp32_train_gemm_mode("tf32x3")
    dev = torch.device("cuda:0")
    shapes = [(76, 100), (38, 50), (19, 25), (10, 13)]

    def pyramid(seed):
        g = torch.Generator().manual_seed(seed)
        return ([torch.randn(2, 256, h, w, generator=g).to(dev, dtype) for h, w in shapes],
                [torch.zeros(2, h, w, dtype=torch.bool, device=dev) for h, w in shapes],
                [torch.randn(2, 256, h, w, generator=g).to(dev, dtype) for h, w in shapes])

    def train():
        torch.manual_seed(11)
        model = DeformableTransformer(num_feature_levels=4, use_depth=True, dropout=0.1,
                                      depth_type="DepthDeform_encoder_cf_dformer").to(dev, dtype).train()
        opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
        srcs, masks, poss = pyramid(1)
        dsrcs, dmasks, dposs = pyramid(2)
        for _ in range(3):
            opt.zero_grad(set_to_none=True)
            src, mask, pos, lv = _flatten_levels(srcs, masks, poss, model.level_embed)
            st, ls = _shape_tensors(lv, dev)
            vr = torch.stack([model.get_valid_ratio(m) for m in masks], 1)
            d_tok, d_mask, d_pos, _, d_st, d_ls, d_vr = model._flatten_depth(dsrcs, dmasks, dposs)
            memory = model.encoder(src, st, ls, vr, pos, mask, None, d_tok, d_st, d_ls, d_vr, d_pos, d_mask)
            memory.float().square().mean().backward()
            opt.step()
        h = hashlib.sha256()
        for p in model.parameters():
            h.update(p.detach().float().cpu().numpy().tobytes())
        return h.hexdigest()

    print("DIGEST", train(), train())
""")


@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_training_is_bitwise_reproducible(dtype):
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8", PYTHONPATH=ROOT)
    proc = subprocess.run([sys.executable, "-c", TRAIN, dtype], cwd=ROOT, env=env, capture_output=True, text=True,
                          timeout=900)
    assert proc.returncode == 0, proc.stdout[-2000:] + proc.stderr[-4000:]
    line = [ln for ln in proc.stdout.splitlines() if ln.startswith("DIGEST")][-1]
    _, first, second = line.split()
    assert first == second, "two training runs from the same seed ended with different parameters"
