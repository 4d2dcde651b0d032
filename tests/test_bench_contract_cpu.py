"""CPU: the reference arm of bench.py (`--impl reference`: the oracle port of the reference's CPU path on the host
cores) prints ONE JSON line with the keys the driver reads, and the algorithmic-byte figures bench.py's roofline uses
are the ones DESIGN.md / SURVEY.md 8(d) state."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

from tests.util import ROOT


def test_reference_arm_prints_the_contract_line(tmp_path):
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                           "--warmup", "1", "--dump-outputs", str(tmp_path)], cwd=ROOT, stdout=subprocess.PIPE,
                          stderr=subprocess.PIPE, text=True, timeout=600)
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [ln for ln in proc.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] == "msda_fwd_bwd_queries_per_sec"
    assert line["unit"] == "queries/s" and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["n_gpus"] == 1 and line["steps"] == 1 and line["warmup"] == 1 and line["value"] > 0
    assert abs(line["value"] - 22223 / (line["ms_per_step"] * 1e-3)) <= 1e-6 * line["value"]   # one frame per step
    assert line["config"]["workload"].startswith("msda_core_op_fwd_bwd") and "model" not in line["config"]
    base = line["cpu_baseline"]
    assert base["kind"] == "port" and base["cores"] >= 1 and base["value"] == line["value"] and base["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "queries/s", "h2d_bytes_per_step": 0,
                           "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0
    # --dump-outputs: the last step's results in float32, 64 MiB at most; a large array is kept at dump_positions()
    sys.path.insert(0, ROOT)
    import bench
    from oracle import msda_oracle
    dumped = {name: np.load(tmp_path / (name + ".npy")) for name in bench.DUMP_NAMES}
    assert sorted(p.name for p in tmp_path.iterdir()) == sorted(n + ".npy" for n in bench.DUMP_NAMES)
    assert all(a.dtype == np.float32 for a in dumped.values())
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64 << 20
    value, loc, attn, _ = bench.make_inputs(torch, 1, 0, "grid")
    out = msda_oracle.core_pytorch(value, bench.COCO_SHAPES, loc, attn).reshape(-1)
    np.testing.assert_allclose(dumped["output"], out[bench.dump_positions(torch, out.numel(), 0)].numpy(),
                               rtol=1e-6, atol=1e-7)
    assert dumped["grad_attn_weight"].shape == tuple(attn.shape)        # small enough to be stored whole


def test_algorithmic_bytes_match_the_stated_per_query_figures():
    sys.path.insert(0, ROOT)
    import bench
    s = sum(h * w for h, w in bench.COCO_SHAPES)
    assert s == 22223
    fwd32, bwd32 = bench.algorithmic_bytes(1, 4)
    fwd16, bwd16 = bench.algorithmic_bytes(1, 2)
    assert (fwd32, bwd32) == (3584 * s, 6144 * s)              # SURVEY.md 8(d): fp32 3584 / 6144 B per query
    # 16-bit values / outputs / gradients, fp32 locations and weights: 512 + 1536 + 512 and 3 x 512 + 2 x 1536 + ... by
    # SURVEY 8(d)'s own formula = 2560 / 4608 B per query (its table prints 4096 for the backward: an addition slip)
    assert (fwd16, bwd16) == (2560 * s, 4608 * s)
