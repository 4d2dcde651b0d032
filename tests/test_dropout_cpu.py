"""CPU: the dropout mask contract (DESIGN.md section 3.16) and its routing.

- The numpy oracle reproduces the Random123 known answers of Philox4x32-10.
- The library's keep rule (threshold, scale) equals the oracle's, and p outside (0, 1) is refused.
- With the library replaced by a recorder, the dropout symbols are called, and a key is drawn, exactly when an
  nn.Dropout is in training with 0 < p < 1 (and PACKAGE_DROPOUT is on); otherwise torch's module runs or nothing does.
"""
import contextlib
import math
import types

import numpy as np
import pytest
import torch
from torch import nn

from dfvod_b200 import _lib
from dfvod_b200.ops.functions import layer_epilogue_func as lef

from .philox_oracle import philox4x32_10, rule


@pytest.mark.parametrize("ctr,key,expected", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, expected):
    r = philox4x32_10(np.array(ctr, dtype=np.uint32), np.array(key, dtype=np.uint32))
    assert tuple(int(v) for v in r) == expected


@pytest.mark.parametrize("p,t", [(0.1, 6554), (0.2, 13107), (0.5, 32768)])
def test_keep_rule_matches_library(p, t):
    assert rule(p)[0] == t
    lib_t, lib_scale = lef.dropout_rule(p)
    assert (lib_t, lib_scale) == rule(p)
    assert lib_scale == float(np.float32(1 / (1 - np.float32(p))))
    assert abs(1 - lib_t / 65536 - (1 - p)) <= 2.0 ** -17


@pytest.mark.parametrize("p", [0.0, 1.0, -0.1, 1.5, math.nan])
def test_keep_rule_refuses_rates_outside_open_interval(p):
    with pytest.raises(_lib.MSDAError):
        lef.dropout_rule(p)


class RecordingLib:
    def __init__(self):
        self.calls = []

    def msda_layer_add_layernorm_supported(self, *args):
        return 1

    def msda_layer_add_layernorm_dropout_supported(self, *args):
        return 1

    def __getattr__(self, name):
        def fn(*args):
            self.calls.append(name)
            return 0
        return fn


class FakeCuda(torch.Tensor):
    """A CPU tensor that reports itself as CUDA, so the routing takes the device path against the recorder."""

    @property
    def is_cuda(self):
        return True


@pytest.fixture
def fake(monkeypatch):
    lib = RecordingLib()
    keys = []
    monkeypatch.setattr(_lib, "_lib", lib)
    monkeypatch.setattr(torch.cuda, "device", lambda *_: contextlib.nullcontext())
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *_: types.SimpleNamespace(cuda_stream=0))
    monkeypatch.setattr(lef, "_dropout_key", lambda device: keys.append(device) or torch.zeros(1, dtype=torch.int64))
    lib.keys = keys
    return lib


class NotExactlyDropout(nn.Dropout):
    pass


# (module, training, package flag, package path expected)
CASES = [
    (nn.Dropout(0.1), True, True, True),
    (nn.Dropout(0.2), True, True, True),
    (nn.Dropout(0.1), False, True, False),
    (nn.Dropout(0.0), True, True, False),
    (nn.Dropout(1.0), True, True, False),
    (nn.Dropout(0.1), True, False, False),
    (NotExactlyDropout(0.1), True, True, False),
]


def _set(module, training, package, monkeypatch):
    module.train(training)
    monkeypatch.setattr(lef, "PACKAGE_DROPOUT", package)


@pytest.mark.parametrize("module,training,package,expected", CASES)
def test_dropout_routing(fake, monkeypatch, module, training, package, expected):
    _set(module, training, package, monkeypatch)
    x = torch.ones(4, 256).as_subclass(FakeCuda)
    lef.dropout(module, x)
    assert ("msda_layer_dropout" in fake.calls) == expected
    assert len(fake.keys) == (1 if expected else 0)


@pytest.mark.parametrize("module,training,package,expected", CASES)
def test_add_layer_norm_routing(fake, monkeypatch, module, training, package, expected):
    _set(module, training, package, monkeypatch)
    norm = nn.LayerNorm(256)
    x = torch.ones(4, 256).as_subclass(FakeCuda)
    lef.add_layer_norm(norm, x, x.clone(), "gelu", dropout=module)
    assert ("msda_layer_add_layernorm_dropout_forward" in fake.calls) == expected
    assert len(fake.keys) == (1 if expected else 0)
    if module.training and module.p > 0 and not expected:
        # torch's module between the kernels: activation and dropout run before the dropout-free norm kernel
        assert fake.calls == ["msda_layer_add_layernorm_forward"]
    if not (module.training and module.p > 0):
        assert fake.calls == ["msda_layer_add_layernorm_forward"]      # the dropout-free path, GELU in the kernel


@pytest.mark.parametrize("module,training,package,expected", CASES)
def test_linear_relu_routing(fake, monkeypatch, module, training, package, expected):
    _set(module, training, package, monkeypatch)
    lin = nn.Linear(256, 64)
    x = torch.ones(4, 256).as_subclass(FakeCuda)
    y = lef.linear_relu(lin, x, module)
    assert y.shape == (4, 64)
    assert ("msda_layer_dropout" in fake.calls) == expected      # library GEMM route: ReLU GEMM + in-place dropout
    assert len(fake.keys) == (1 if expected else 0)
