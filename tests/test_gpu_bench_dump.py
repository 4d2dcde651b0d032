"""GPU: bench.py --dump-outputs writes what the timed op returned in its last timed step, at the positions
bench.dump_positions names, so two builds run with the same arguments can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.util import ROOT

pytestmark = pytest.mark.gpu


def test_b200_arm_dumps_the_last_timed_step(tmp_path):
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--batch", "1",
                           "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], cwd=ROOT,
                          stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [ln for ln in proc.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64 << 20

    sys.path.insert(0, ROOT)
    import bench
    from dfvod_b200 import MultiScaleDeformableAttention as MSDA
    value, loc, attn, gout = (t.cuda() for t in bench.make_inputs(torch, 1, 1000, "grid"))   # rank 0's inputs
    st = torch.as_tensor(bench.COCO_SHAPES, dtype=torch.long, device="cuda")
    ls = torch.as_tensor(bench.level_start(bench.COCO_SHAPES)[0], dtype=torch.long, device="cuda")
    want = (MSDA.ms_deform_attn_forward(value, st, ls, loc, attn, 64),
            *MSDA.ms_deform_attn_backward(value, st, ls, loc, attn, gout, 64))
    for seed, (name, w) in enumerate(zip(bench.DUMP_NAMES, want)):
        got = np.load(tmp_path / (name + ".npy"))
        assert got.dtype == np.float32
        if w.numel() > bench.DUMP_SAMPLE:
            w = w.reshape(-1)[bench.dump_positions(torch, w.numel(), seed).cuda()]
        w = w.float().cpu().numpy()
        assert got.shape == w.shape, name
        if name == "grad_value":            # accumulated with atomics: order-dependent rounding only
            assert np.abs(got - w).max() <= 1e-5 * np.abs(w).max(), name
        else:
            np.testing.assert_array_equal(got, w, err_msg=name)
