"""CPU: the backward of the plain op, the fused op and RoIAlign calls the *_deterministic symbol exactly when
torch.are_deterministic_algorithms_enabled() (warn_only included), with a scratch of the size the library asks for.
The library is replaced by a recorder, so no GPU is needed."""
import contextlib
import types

import pytest
import torch

from dfvod_b200 import _lib
from dfvod_b200 import MultiScaleDeformableAttention as MSDA
from dfvod_b200 import temporal_stage
from dfvod_b200.ops.functions import MSDeformAttnFusedFunction


class RecordingLib:
    SCRATCH = 96

    def __init__(self):
        self.calls = []

    def msda_deterministic_scratch_bytes(self, *args):
        self.calls.append(("msda_deterministic_scratch_bytes", args))
        return self.SCRATCH

    def __getattr__(self, name):
        def fn(*args):
            self.calls.append((name, args))
            return 0
        return fn

    def names(self):
        return [c[0] for c in self.calls]


@pytest.fixture
def fake(monkeypatch):
    lib = RecordingLib()
    monkeypatch.setattr(_lib, "_lib", lib)
    monkeypatch.setattr(torch.cuda, "device", lambda *_: contextlib.nullcontext())
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *_: types.SimpleNamespace(cuda_stream=0))
    monkeypatch.setattr(MSDA, "_check_inputs", lambda *_: None)
    return lib


@contextlib.contextmanager
def flag(on, warn_only=False):
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(on, warn_only=warn_only)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_warn)


MODES = [(False, False, False), (True, False, True), (True, True, True)]      # (flag, warn_only, deterministic?)


@pytest.mark.parametrize("on,warn_only,det", MODES)
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_plain_op_routing(fake, on, warn_only, det, dtype):
    n, s, m, d, nl, lq, p = 1, 6, 2, 4, 1, 3, 2
    value = torch.zeros(n, s, m, d, dtype=dtype)
    shapes, lsi = torch.tensor([[2, 3]]), torch.tensor([0])
    loc, attn = torch.zeros(n, lq, m, nl, p, 2), torch.zeros(n, lq, m, nl, p)
    with flag(on, warn_only):
        MSDA.ms_deform_attn_backward(value, shapes, lsi, loc, attn, torch.zeros(n, lq, m * d, dtype=dtype), 64)
    names = fake.names()
    if det:
        assert names == ["msda_deterministic_scratch_bytes", "msda_backward_deterministic"]
        assert fake.calls[0][1] == (value.numel(), 0, 0)
        args = fake.calls[1][1]
        assert args[-2] == RecordingLib.SCRATCH and args[-5] is None      # scratch size; no fp32 accumulator
    else:
        assert names == ["msda_backward"]


@pytest.mark.parametrize("on,warn_only,det", MODES)
@pytest.mark.parametrize("ref_grad", [True, False])
def test_fused_op_routing(fake, on, warn_only, det, ref_grad):
    n, s, m, d, nl, lq, p = 1, 6, 2, 4, 1, 3, 2
    value = torch.zeros(n, s, m, d, requires_grad=True)
    raw = torch.zeros(n, lq, 3 * m * nl * p, requires_grad=True)
    ref = torch.zeros(n, lq, nl, 2, requires_grad=ref_grad)
    out = MSDeformAttnFusedFunction.apply(value, torch.tensor([[2, 3]]), torch.tensor([0]), ref, raw, p)
    fake.calls.clear()
    with flag(on, warn_only):
        out.backward(torch.zeros_like(out))
    names = fake.names()
    if det:
        assert names == ["msda_deterministic_scratch_bytes", "msda_fused_backward_deterministic"]
        assert fake.calls[0][1] == (value.numel(), ref.numel() if ref_grad else 0, m)
    else:
        assert names == ["msda_fused_backward"]
    assert (ref.grad is not None) == ref_grad


@pytest.mark.parametrize("on,warn_only,det", MODES)
def test_roi_align_routing(fake, on, warn_only, det):
    n, h, w, c, k = 2, 3, 4, 8, 5
    ctx = types.SimpleNamespace(saved_tensors=(torch.zeros(k, 5),),
                                geom=(n, h, w, c, 7, 7, 1.0, 2, 1, torch.bfloat16))
    with flag(on, warn_only):
        grads = temporal_stage._RoIAlignTokens.backward(ctx, torch.zeros(k, 49, c, dtype=torch.bfloat16))
    names = fake.names()
    assert grads[0].shape == (n, h * w, c) and grads[0].dtype == torch.bfloat16
    if det:
        assert names == ["msda_deterministic_scratch_bytes", "msda_roi_align_backward_deterministic"]
        assert fake.calls[0][1] == (n * h * w * c, 0, 0)
    else:
        assert names == ["msda_roi_align_backward"]
