#!/usr/bin/env python
"""Benchmark of the MSDeformAttn hot path (BASELINE.json metric: "MSDeformAttn fwd+bwd
queries/sec & HBM GB/s vs roofline").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                  [--dtype f32|bf16] [--dist grid|random] [--batch B] [--dump-outputs DIR]

One "step" = one forward + one backward of the drop-in op
``MSDeformAttnFunction`` (C ABI msda_forward + msda_backward) over one batch of B=8 frames of
the COCO-scale 4-level pyramid of an 800x1333 input (S = Lq = 22223 tokens per frame, M=8
heads, D=32, L=4, P=4): the encoder self-attention shape of BASELINE.json configs[1].
Inputs of one step are 637 MB (fp32) > the 126 MB L2, so no explicit L2 flush is needed.
N>1: one process per GPU (torchrun), every rank runs its own batch (frames shard across GPUs,
no data-path collective) -> weak scaling; time = max over ranks.

``--impl reference`` times the reference's CPU implementation of the same path -- the in-repo
restatement of ms_deform_attn_core_pytorch (oracle/msda_oracle.py; the original cannot be
imported on the GPU box, /root/reference does not travel) -- fwd + autograd bwd, all host
threads, on a bounded sample (1 frame per step).

``--dump-outputs DIR`` writes what the timed op returned in its last timed step (rank 0) as
DIR/<name>.npy in float32: output, grad_value, grad_sampling_loc, grad_attn_weight.  An array of
more than DUMP_SAMPLE elements is stored as the elements at DUMP_SAMPLE fixed positions drawn from
a seeded generator (the same positions in every run), so two builds run with the same arguments
can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the source tree as it found it

COCO_SHAPES = [(100, 167), (50, 84), (25, 42), (13, 21)]
M, D, P = 8, 32, 4
METRIC = "msda_fwd_bwd_queries_per_sec"
UNIT = "queries/s"
DUMP_NAMES = ("output", "grad_value", "grad_sampling_loc", "grad_attn_weight")
DUMP_SAMPLE = 3 << 20                   # elements kept per array: 4 arrays x 12 MiB of float32 <= 64 MiB


def level_start(shapes):
    out, acc = [], 0
    for h, w in shapes:
        out.append(acc)
        acc += h * w
    return out, acc


def make_inputs(torch, n, seed, dist):
    """CPU generator (identical bits for the CPU arm and the GPU arm)."""
    import math
    g = torch.Generator().manual_seed(seed)
    lsi, s = level_start(COCO_SHAPES)
    nl, lq = len(COCO_SHAPES), s
    value = torch.randn(n, s, M, D, generator=g)
    attn = torch.softmax(torch.randn(n, lq, M, nl * P, generator=g), -1).view(n, lq, M, nl, P)
    if dist == "random":                       # reference test recipe: loc ~ U[0,1)  (models/ops/test.py:34)
        loc = torch.rand(n, lq, M, nl, P, 2, generator=g)
    else:                                      # encoder geometry: pixel-centre grid + init compass offsets + N(0,1) px
        ref = []
        for h, w in COCO_SHAPES:
            ys = (torch.arange(h, dtype=torch.float32) + 0.5) / h
            xs = (torch.arange(w, dtype=torch.float32) + 0.5) / w
            yy, xx = torch.meshgrid(ys, xs, indexing="ij")
            ref.append(torch.stack([xx.reshape(-1), yy.reshape(-1)], -1))
        ref = torch.cat(ref, 0)
        ang = torch.arange(M, dtype=torch.float32) * (2.0 * math.pi / M)
        comp = torch.stack([ang.cos(), ang.sin()], -1)
        comp = comp / comp.abs().max(-1, keepdim=True)[0]
        steps = torch.arange(1, P + 1, dtype=torch.float32)
        off = comp[:, None, None, :] * steps[None, None, :, None]
        noise = torch.randn(n, lq, M, nl, P, 2, generator=g)
        if dist == "init":                     # a freshly initialised layer: offsets are the compass pattern exactly
            noise = noise * 0.0
        off = off.expand(M, nl, P, 2) + noise
        norm = torch.tensor([[w, h] for h, w in COCO_SHAPES], dtype=torch.float32)
        loc = ref[None, :, None, None, None, :] + off / norm[None, None, None, :, None, :]
    grad_out = torch.randn(n, lq, M * D, generator=g)
    return value.contiguous(), loc.contiguous(), attn.contiguous(), grad_out.contiguous()


def dump_positions(torch, numel, seed):
    """The flat positions --dump-outputs keeps of an array of more than DUMP_SAMPLE elements: sorted, drawn from a
    generator seeded by the array's place in DUMP_NAMES, so they depend on the array's size alone."""
    return torch.randint(numel, (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(seed)).sort().values


def dump_outputs(torch, path, arrays):
    """Write the op's results (in DUMP_NAMES order) as <path>/<name>.npy in float32; an array of more than
    DUMP_SAMPLE elements is written flat, as its elements at dump_positions()."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for seed, (name, t) in enumerate(zip(DUMP_NAMES, arrays)):
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            t = t.reshape(-1)[dump_positions(torch, t.numel(), seed).to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.float().cpu().numpy())


def algorithmic_bytes(n, e_v):
    """SURVEY.md 8(d): every operand of the drop-in op counted once.  e_v = bytes per element of
    value / output / grad_output / grad_value; locations and attention weights are fp32."""
    _, s = level_start(COCO_SHAPES)
    lq, c, nl = s, M * D, len(COCO_SHAPES)
    side = lq * M * nl * P * (2 * 4 + 4)
    fwd = n * (s * c * e_v + side + lq * c * e_v)
    bwd = n * (s * c * e_v + side + lq * c * e_v + s * c * e_v + side)
    return fwd, bwd


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md).  Uses NVML
    in-process (a polling `nvidia-smi -lms` child was measured to stall individual launches by
    10-30 ms on this box); falls back to one nvidia-smi query per sample if pynvml is missing."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
               ("sw_power_cap", 0x4))

    def __init__(self, index, period_s=0.05):
        self.index, self.period, self.rows = index, period_s, []
        self._stop = threading.Event()
        self.thread = None
        self.nvml = None

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.index])
            except Exception:
                pass
        return self.index

    def __enter__(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nvml = None
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()
        return self

    def _sample(self):
        if self.nvml is not None:
            n = self.nvml
            sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
            try:
                mask = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
            except Exception:
                mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
            power = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
            return float(sm), float(self.max_sm), power, [name for name, bit in self.REASONS if mask & bit]
        out = subprocess.run(
            ["nvidia-smi", "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-i", str(self._physical_index())],
            stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=10).stdout
        r = [x.strip() for x in out.strip().split(",")]
        return float(r[0]), float(r[1]), float(r[2]), [name for (name, _), flag in zip(self.REASONS, r[3:7])
                                                      if flag.lower().startswith("active")]

    def _pump(self):
        while not self._stop.is_set():
            try:
                self.rows.append(self._sample())
            except Exception:
                pass
            self._stop.wait(self.period)

    def __exit__(self, *exc):
        self._stop.set()
        if self.thread is not None:
            self.thread.join(timeout=5)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(r[0] for r in self.rows)
        reasons = sorted({name for r in self.rows for name in r[3]})
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(r[1] for r in self.rows), "reasons": reasons,
                "samples": len(sm), "power_w_max": max(r[2] for r in self.rows),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def traffic_from_profile(kind, dtype="f32"):
    """dram__bytes_read+write per launch of the kernel from the committed ncu capture
    (profiles/ncu_summary.json, same workload), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_summary.json")) as f:
            return json.load(f).get(dtype, {}).get(kind, {}).get("dram_bytes_per_launch")
    except Exception:
        return None


def profile_build_matches():
    """True when profiles/ncu_summary.json was captured from the gather-kernel sources this library is built from
    (tools/build_hash.py), False when the sources changed since, None when unknown."""
    try:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import build_hash
        with open(os.path.join(ROOT, "profiles", "ncu_summary.json")) as f:
            stamp = json.load(f).get("gather_kernels_build", {}).get("sha256_16")
        return None if stamp is None else stamp == build_hash.gather_kernels_hash()
    except Exception:
        return None


def limiter_from_profile(kind, dtype="f32"):
    """The on-chip unit that bounds the kernel, from the committed ncu capture (DESIGN.md section 3):
    the gather kernels are not HBM-bound -- the forward saturates the L1 data pipe (128 B/clk/SM), the backward the L1
    data pipe and the L1 -> crossbar request path its vector reductions leave the SM through."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_summary.json")) as f:
            k = json.load(f).get(dtype, {}).get(kind, {})
        if kind == "forward":
            return {"unit": "L1 data pipe (l1tex__data_pipe_lsu_wavefronts, 128 B/clk/SM)",
                    "busy_pct": k.get("l1_data_pipe_pct"), "source": "profiles/ncu_summary.json"}
        # two units sit within a few points of each other: report the busier one and keep the other beside it
        units = {"L1 data pipe (l1tex__data_pipe_lsu_wavefronts, 128 B/clk/SM: loads, reductions, records, shuffles)":
                     k.get("l1_data_pipe_pct"),
                 "L1->crossbar request path (l1tex__m_l1tex2xbar_req_cycles_active; RED packets)":
                     k.get("l1_to_xbar_req_busy_pct")}
        top = max(units, key=lambda u: units[u] or 0.0)
        other = [u for u in units if u != top][0]
        return {"unit": top, "busy_pct": units[top], "next": {"unit": other, "busy_pct": units[other]},
                "source": "profiles/ncu_summary.json"}
    except Exception:
        return None


# ----------------------------------------------------------------------------------------------
# CPU arm: the reference's ms_deform_attn_core_pytorch (restated), fwd + autograd bwd
# ----------------------------------------------------------------------------------------------
def time_cpu_reference(torch, steps, warmup, dist, seed=0):
    from oracle import msda_oracle
    torch.set_num_threads(os.cpu_count() or 1)
    value, loc, attn, gout = make_inputs(torch, 1, seed, dist)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        outputs = msda_oracle.core_pytorch_fwd_bwd(value, COCO_SHAPES, loc, attn, gout)
        times.append(time.perf_counter() - t0)
    timed = times[warmup:]
    total = sum(timed)
    q = value.shape[1] * len(timed)
    return {"value": q / total, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{len(timed)} x (1 frame, {value.shape[1]} queries) fwd+bwd, fp32, "
                      f"oracle.core_pytorch (= reference ms_deform_attn_core_pytorch) + autograd, "
                      f"os.cpu_count()={os.cpu_count()}",
            "ms_per_step": 1e3 * total / len(timed), "outputs": outputs}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    cb = time_cpu_reference(torch, args.steps, max(args.warmup, 1), args.dist)
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": cb["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": "msda_core_op_fwd_bwd_coco_pyramid_800x1333", "levels": COCO_SHAPES,
                       "queries_per_frame": level_start(COCO_SHAPES)[1], "heads": M, "head_dim": D,
                       "points": P, "frames_per_step": 1, "loc_distribution": args.dist,
                       "note": "bounded sample: 1 frame per step on host cores"},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if args.dump_outputs:
        dump_outputs(torch, args.dump_outputs, cb["outputs"])
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def _time_events(torch, fn, iters, warm):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def _reduce_max(torch, dist, world, dev, ms):
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def _graph_time(torch, fn, iters):
    """Capture fn() in a CUDA graph (dfvod_b200.data_parallel.GraphedInference) and time the replay."""
    from dfvod_b200.data_parallel import GraphedInference
    run = GraphedInference(fn)
    return _time_events(torch, run, iters, 3)


def _pyramid(torch, dev, shapes, n, dtype, seed):
    g = torch.Generator().manual_seed(seed)
    srcs = [torch.randn(n, 256, h, w, generator=g).to(dev, dtype) for h, w in shapes]
    pos = [torch.randn(n, 256, h, w, generator=g).to(dev, dtype) for h, w in shapes]
    masks = [torch.zeros(n, h, w, dtype=torch.bool, device=dev) for h, w in shapes]
    return srcs, masks, pos


def encoder_extras(torch, dev, world, dist, n_frames=8, iters=10):
    """BASELINE.json "encoder frames/sec" and configs[1]: Deformable DETR single-frame 6+6
    transformer, inference, synthetic ResNet-50-shaped features of an 800x1333 image (4 levels,
    22223 tokens), batch 8 per GPU, 300 queries.  bf16 weights/activations, CUDA-graph replay;
    fp32 (the reference's dtype) for the encoder alone."""
    from dfvod_b200 import transformer_layers as tl
    from dfvod_b200.deformable_transformer import DeformableTransformer
    lsi, s = level_start(COCO_SHAPES)
    st = torch.as_tensor(COCO_SHAPES, dtype=torch.long, device=dev)
    ls = torch.as_tensor(lsi, dtype=torch.long, device=dev)
    torch.manual_seed(1)
    model = DeformableTransformer(num_feature_levels=4, return_intermediate_dec=True).to(dev).eval()
    out = {"frames_per_gpu": n_frames, "tokens_per_frame": s, "queries": 300,
           "model": "DeformableTransformer(d_model=256, 6 enc + 6 dec, 4 levels)"}
    with torch.no_grad():
        src = torch.randn(n_frames, s, 256, device=dev)
        pos = torch.randn(n_frames, s, 256, device=dev)
        vr = torch.ones(n_frames, len(COCO_SHAPES), 2, device=dev)
        from dfvod_b200.ops.functions import set_fp32_gemm_mode
        # fp32 as the package runs it by default: fp32-grade GEMMs on the tensor cores (three-term TF32 split inside one
        # tcgen05 kernel, csrc/linear_tf32x3.cu; <= 7e-7 normalised against fp64 per GEMM at K = 256 -- the IEEE SGEMM's
        # own error), gathers in fp32
        ms = _reduce_max(torch, dist, world, dev,
                         _time_events(torch, lambda: model.encoder(src, st, ls, vr, pos, None), 3, 2))
        out["encoder_fp32_ms"] = ms
        out["encoder_fp32_fps"] = n_frames * world / ms * 1e3
        out["encoder_fp32_gemm_mode"] = "tf32x3 (dfvod_b200.ops.functions.set_fp32_gemm_mode default)"
        try:                                       # the same fp32 encoder replayed from one CUDA graph, like the bf16 lines
            ms = _reduce_max(torch, dist, world, dev,
                             _graph_time(torch, lambda: model.encoder(src, st, ls, vr, pos, None), 3))
            out["encoder_fp32_graph_ms"] = ms
            out["encoder_fp32_graph_fps"] = n_frames * world / ms * 1e3
        except Exception as exc:
            out["encoder_fp32_graph_error"] = repr(exc)[:160]
        # the same encoder with the library's IEEE SGEMMs (set_fp32_gemm_mode("library"): the reference's own arithmetic)
        prev_mode = set_fp32_gemm_mode("library")
        try:
            ms = _reduce_max(torch, dist, world, dev,
                             _time_events(torch, lambda: model.encoder(src, st, ls, vr, pos, None), 3, 2))
            out["encoder_fp32_ieee_gemm_ms"] = ms
            out["encoder_fp32_ieee_gemm_fps"] = n_frames * world / ms * 1e3
            # ... and with the library GEMMs allowed to use plain TF32 (the caller's opt-in,
            # torch.backends.cuda.matmul.allow_tf32).  Not parity-grade: 3e-4 per GEMM.
            prev_tf32 = torch.backends.cuda.matmul.allow_tf32
            torch.backends.cuda.matmul.allow_tf32 = True
            try:
                ms = _reduce_max(torch, dist, world, dev,
                                 _time_events(torch, lambda: model.encoder(src, st, ls, vr, pos, None), 3, 2))
                out["encoder_fp32_tf32_gemm_ms"] = ms
                out["encoder_fp32_tf32_gemm_fps"] = n_frames * world / ms * 1e3
            finally:
                torch.backends.cuda.matmul.allow_tf32 = prev_tf32
        finally:
            set_fp32_gemm_mode(prev_mode)
        del src, pos
        model = model.bfloat16()
        bf = torch.bfloat16
        src16 = torch.randn(n_frames, s, 256, device=dev, dtype=bf)
        pos16 = torch.randn(n_frames, s, 256, device=dev, dtype=bf)
        enc = lambda: model.encoder(src16, st, ls, vr, pos16, None)
        ms = _reduce_max(torch, dist, world, dev, _time_events(torch, enc, iters, 3))
        out["encoder_bf16_eager_fps"] = n_frames * world / ms * 1e3
        try:
            ms = _reduce_max(torch, dist, world, dev, _graph_time(torch, enc, iters))
            out["encoder_bf16_graph_ms"] = ms
            out["encoder_bf16_graph_fps"] = n_frames * world / ms * 1e3
        except Exception as exc:      # report, do not hide
            out["encoder_bf16_graph_error"] = repr(exc)[:160]
        del src16, pos16
        srcs, masks, poss = _pyramid(torch, dev, COCO_SHAPES, n_frames, bf, 2)
        query = torch.randn(300, 512, device=dev, dtype=bf)
        full = lambda: model(srcs, masks, poss, None, None, None, query)
        ms = _reduce_max(torch, dist, world, dev, _time_events(torch, full, iters, 3))
        out["enc_dec_bf16_eager_fps"] = n_frames * world / ms * 1e3
        try:
            ms = _reduce_max(torch, dist, world, dev, _graph_time(torch, full, iters))
            out["enc_dec_bf16_graph_ms"] = ms
            out["enc_dec_bf16_graph_fps"] = n_frames * world / ms * 1e3
        except Exception as exc:
            out["enc_dec_bf16_graph_error"] = repr(exc)[:160]
    return out


def clip_extras(torch, dev, world, dist, iters=10):
    """BASELINE.json configs[3]: TransVOD++ multi-frame encoder with Late Fusion, inference.  A clip =
    1 current + 3 reference frames = batch 4 (frames of a clip are the batch dimension of every
    MSDeformAttn call, deformable_transformer_multi_plusplus.py:260-444); one feature level
    (50,84) as in the shipped configs; 8 clips per GPU per step; transformer = Late-Fusion layer +
    6 encoder + 6 decoder layers, bf16, CUDA graph.  (The temporal query stage is out of scope.)"""
    from dfvod_b200.deformable_transformer import DeformableTransformer
    shapes, clip, clips = [(50, 84)], 4, 8
    torch.manual_seed(3)
    model = DeformableTransformer(num_feature_levels=1, return_intermediate_dec=True, use_depth=True,
                                  depth_type="DepthDeform_latefusion_dformer").to(dev).eval().bfloat16()
    bf = torch.bfloat16
    n = clip * clips
    with torch.no_grad():
        srcs, masks, poss = _pyramid(torch, dev, shapes, n, bf, 5)
        dsrcs, dmasks, dposs = _pyramid(torch, dev, shapes, n, bf, 6)
        query = torch.randn(300, 512, device=dev, dtype=bf)
        run = lambda: model(srcs, masks, poss, dsrcs, dmasks, dposs, query)
        ms = _reduce_max(torch, dist, world, dev, _time_events(torch, run, iters, 3))
        out = {"clip_frames": clip, "clips_per_gpu": clips, "level": shapes[0], "eager_fps": n * world / ms * 1e3}
        try:
            ms = _reduce_max(torch, dist, world, dev, _graph_time(torch, run, iters))
            out["graph_ms"] = ms
            out["graph_fps"] = n * world / ms * 1e3
        except Exception as exc:
            out["graph_error"] = repr(exc)[:160]
        del model
        try:
            out["with_temporal_stage"] = _clip_temporal(torch, dev, world, dist, shapes, clip, clips, iters,
                                                        (srcs, masks, poss, dsrcs, dmasks, dposs, query))
        except Exception as exc:      # report, do not hide
            out["with_temporal_stage"] = {"error": repr(exc)[:200]}
    return out


def _clip_temporal(torch, dev, world, dist, shapes, clip, clips, iters, inputs):
    """The same clips through the WHOLE TransVOD++ transformer (dfvod_b200.temporal_stage.DeformableTransformer):
    per-frame Late Fusion + encoder + decoder with box refinement, then the temporal query stage -- RoIAlign of all
    300 boxes of every frame (csrc/roi_align.cu), QRF head, 3 x (temporal query encoder + temporal deformable
    decoder); 8 clips batched clip-major, detection heads with random weights, 31 classes, bf16."""
    from torch import nn
    from dfvod_b200 import temporal_stage
    bf = torch.bfloat16
    torch.manual_seed(33)
    tr = temporal_stage.DeformableTransformer(
        num_feature_levels=1, return_intermediate_dec=True, use_depth=True, num_ref_frames=clip - 1,
        depth_type="DepthDeform_latefusion_dformer")

    def mlp():
        return nn.Sequential(nn.Linear(256, 256), nn.ReLU(), nn.Linear(256, 256), nn.ReLU(), nn.Linear(256, 4))

    heads = nn.ModuleDict(dict(cls=nn.Linear(256, 31), box=nn.ModuleList(mlp() for _ in range(6)),
                               tcls=nn.ModuleList(nn.Linear(256, 31) for _ in range(3)),
                               tbox=nn.ModuleList(mlp() for _ in range(3))))
    tr.decoder.bbox_embed = heads["box"]                      # --with_box_refine, as TransVOD++ is trained
    tr = tr.to(dev).eval().to(bf)
    heads = heads.to(dev).eval().to(bf)
    srcs, masks, poss, dsrcs, dmasks, dposs, query = inputs
    h, w = shapes[0]
    whwh = torch.tensor([[w * 32, h * 32, w * 32, h * 32]], dtype=torch.long, device=dev)
    n = clip * clips
    run = lambda: tr(srcs, masks, poss, dsrcs, dmasks, dposs, whwh, query, heads["cls"], heads["box"][-1],
                     heads["tcls"], heads["tbox"])
    ms = _reduce_max(torch, dist, world, dev, _time_events(torch, run, iters, 3))
    out = {"eager_ms": ms, "eager_fps": n * world / ms * 1e3, "eager_clips_per_s": clips * world / ms * 1e3}
    try:
        ms = _reduce_max(torch, dist, world, dev, _graph_time(torch, run, iters))
        out.update(graph_ms=ms, graph_fps=n * world / ms * 1e3, graph_clips_per_s=clips * world / ms * 1e3)
    except Exception as exc:
        out["graph_error"] = repr(exc)[:160]
    # the RoIAlign kernel alone at this size (8 clips x 4 frames x 300 boxes, 7x7x256 out of a 50x84 map)
    tokens = torch.randn(n, h * w, 256, device=dev, dtype=bf)
    g = torch.Generator().manual_seed(5)
    cxy = torch.rand(n * 300, 2, generator=g) * torch.tensor([w * 32.0, h * 32.0])
    wh = torch.rand(n * 300, 2, generator=g) * torch.tensor([w * 16.0, h * 16.0]) + 8
    rois = torch.cat([torch.arange(n).repeat_interleave(300)[:, None].float(), cxy - wh / 2, cxy + wh / 2], -1).to(dev)
    ms = _time_events(torch, lambda: temporal_stage.roi_align_tokens(tokens, rois, h, w, 7, 1 / 32, 2, True), 20, 3)
    out["roi_align_kernel"] = {"rois": n * 300, "ms": ms, "output_gbytes_per_s": n * 300 * 49 * 256 * 2 / ms / 1e6}
    return out


def fusion_layer_extras(torch, dev, world, dist, n_frames=4, iters=10):
    """BASELINE.json configs[2]: Encoder Cross Fusion RGB-D -- RGB queries deformably attending to the depth
    feature pyramid -- one DeformableTransformerFusionLayerV2, forward + backward, bf16, batch 4 frames per GPU
    (Encoder_CrossFusion.sh:18).  (i) as shipped: one level (50,84); (ii) COCO scale: the 4-level pyramid."""
    from dfvod_b200 import transformer_layers as tl
    out = {"frames_per_gpu": n_frames, "dtype": "bf16"}
    bf = torch.bfloat16
    for tag, shapes in (("shipped_1_level_50x84", [(50, 84)]), ("coco_4_levels", COCO_SHAPES)):
        lsi, s = level_start(shapes)
        st = torch.as_tensor(shapes, dtype=torch.long, device=dev)
        ls = torch.as_tensor(lsi, dtype=torch.long, device=dev)
        torch.manual_seed(2)
        layer = tl.DeformableTransformerFusionLayerV2(256, 1024, 0.0, "gelu", len(shapes), 8, 4).to(dev).to(bf)
        g = torch.Generator().manual_seed(2)
        tgt = torch.randn(n_frames, s, 256, generator=g).to(dev, bf).requires_grad_(True)
        qpos = torch.randn(n_frames, s, 256, generator=g).to(dev, bf)
        src = torch.randn(n_frames, s, 256, generator=g).to(dev, bf).requires_grad_(True)
        ref = tl.encoder_reference_points(shapes, torch.ones(n_frames, len(shapes), 2, device=dev), dev)

        def step():
            loss = layer(tgt, qpos, ref, src, st, ls, None).float().square().mean()
            loss.backward()
            layer.zero_grad(set_to_none=True)
            tgt.grad = src.grad = None

        ms = _reduce_max(torch, dist, world, dev, _time_events(torch, step, iters, 3))
        out[tag] = {"tokens_per_frame": s, "fwd_bwd_ms": ms, "frames_per_s": n_frames * world / ms * 1e3}
        del layer, tgt, qpos, src, ref
    return out


def input_projection_extras(torch, dev, world, dist, n_frames=8, iters=10):
    """SURVEY.md 8f rank 4: the input projections in front of the transformer (Conv2d 1x1 + GroupNorm(32, 256) per
    backbone level, deformable_detr_single.py:101-150) on ResNet-50-shaped features of an 800x1333 image (C3 512 ch
    100x167, C4 1024 ch 50x84, C5 2048 ch 25x42), batch 8, bf16: the reference's composition (NCHW conv, GroupNorm,
    flatten + transpose + cat to tokens) against InputProjection.forward_tokens (token-major GEMM + in-place token
    GroupNorm kernels)."""
    from dfvod_b200.input_projection import InputProjection
    bf = torch.bfloat16
    levels = [(512, 100, 167), (1024, 50, 84), (2048, 25, 42)]
    torch.manual_seed(8)
    projs = [InputProjection(cin, 256).to(dev).to(bf).eval() for cin, _, _ in levels]
    feats = [torch.randn(n_frames, cin, h, w, device=dev).to(bf) for cin, h, w in levels]
    with torch.no_grad():
        composition = lambda: torch.cat([p(x).flatten(2).transpose(1, 2) for p, x in zip(projs, feats)], 1)
        from dfvod_b200.input_projection import project_levels
        tokens = lambda: project_levels(projs, feats)[0]
        ms_ref = _reduce_max(torch, dist, world, dev, _time_events(torch, composition, iters, 3))
        ms_tok = _reduce_max(torch, dist, world, dev, _time_events(torch, tokens, iters, 3))
        gn_in = torch.randn(n_frames, 16700, 256, device=dev).to(bf)
        from dfvod_b200.input_projection import group_norm_tokens
        norm = projs[0][1]
        ms_gn = _time_events(torch, lambda: group_norm_tokens(gn_in, 32, norm.weight, norm.bias, 1e-5, inplace=True), 20, 3)
        # sine position embedding of the 4-level pyramid + level embedding -> lvl_pos_embed_flatten
        # (position_encoding.py:35-56, backbone_scratch.py:185, deformable_transformer_single.py:196-206)
        from dfvod_b200.position_encoding import PositionEmbeddingSine
        sine = PositionEmbeddingSine(128, normalize=True)
        masks = [torch.zeros(n_frames, h, w, dtype=torch.bool, device=dev) for h, w in COCO_SHAPES]
        lvl_embed = torch.randn(len(COCO_SHAPES), 256, device=dev).to(bf)
        pos_ref = lambda: torch.cat([sine._host_composition(m).permute(0, 3, 1, 2).to(bf).flatten(2).transpose(1, 2)
                                     + lvl_embed[i].view(1, 1, -1) for i, m in enumerate(masks)], 1)
        pos_tok = lambda: sine.forward_tokens(masks, lvl_embed, dtype=bf)
        ms_pos_ref = _time_events(torch, pos_ref, iters, 3)
        ms_pos_tok = _time_events(torch, pos_tok, iters, 3)
    gn_bytes = gn_in.numel() * 2 * 3                       # read (statistics), read + write (apply)
    return {"frames_per_gpu": n_frames, "levels": levels, "dtype": "bf16", "reference_composition_ms": ms_ref,
            "token_major_ms": ms_tok,
            "sine_position_tokens": {"tokens_per_frame": sum(h * w for h, w in COCO_SHAPES),
                                     "reference_composition_ms": ms_pos_ref, "kernel_ms": ms_pos_tok},
            "group_norm_tokens_kernels": {"rows": n_frames * 16700, "ms": ms_gn, "gbytes_per_s": gn_bytes / ms_gn / 1e6}}


def train_step_extras(torch, dev, world, dist, n_frames=4, iters=5):
    """BASELINE.json configs[4]: Encoder-Cross-Fusion training step (fwd + bwd + AdamW), frames
    sharded over GPUs, gradients all-reduced over NCCL by dfvod_b200.data_parallel.  Model:
    DeformableTransformer(depth_type='DepthDeform_encoder_cf_dformer') = 6 encoder + 4 fusion + 6
    decoder layers, COCO pyramid for RGB and for depth, 300 queries, bf16 parameters, synthetic
    features, loss = mean(hs^2)."""
    from dfvod_b200 import data_parallel
    from dfvod_b200.deformable_transformer import DeformableTransformer
    torch.manual_seed(4)                      # identical initial weights on every rank
    model = DeformableTransformer(num_feature_levels=4, return_intermediate_dec=True, use_depth=True, dropout=0.0,
                                  depth_type="DepthDeform_encoder_cf_dformer").to(dev).bfloat16()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-5, fused=True)
    reducer = data_parallel.GradientAllReducer(model.parameters())
    rank = dist.get_rank() if world > 1 else 0
    bf = torch.bfloat16
    srcs, masks, poss = _pyramid(torch, dev, COCO_SHAPES, n_frames, bf, 40 + rank)
    dsrcs, dmasks, dposs = _pyramid(torch, dev, COCO_SHAPES, n_frames, bf, 140 + rank)
    query = torch.randn(300, 512, generator=torch.Generator().manual_seed(7)).to(dev, bf)

    def step():
        opt.zero_grad(set_to_none=True)
        hs = model(srcs, masks, poss, dsrcs, dmasks, dposs, query)[0]
        loss = hs.float().square().mean()
        loss.backward()
        reducer.finish()
        opt.step()
        return loss

    def params_agree():
        """SURVEY.md C5: after data-parallel steps every rank must hold the same parameters.  Compares the
        element-wise MIN and MAX over ranks of every parameter (one flat fp32 vector); on one GPU trivially true."""
        flat = torch.cat([p.detach().float().flatten() for p in model.parameters()])
        if world == 1:
            return True, 0.0
        lo, hi = flat.clone(), flat.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        return bool(torch.equal(lo, hi)), float((hi - lo).abs().max().item())

    ms = _reduce_max(torch, dist, world, dev, _time_events(torch, step, iters, 2))
    reducer.remove()
    same, spread = params_agree()
    assert same, f"parameters differ across ranks after the eager data-parallel steps (max spread {spread:.3e})"
    out = {"frames_per_gpu": n_frames, "eager_ms_per_step": ms, "eager_frames_per_s": n_frames * world / ms * 1e3,
           "gradient_bytes": reducer.gradient_bytes, "dtype": "bf16",
           "collective": "bucketed all-reduce (NCCL)" if world > 1 else "none (1 GPU)",
           "params_equal_across_ranks_after_eager_steps": same}
    try:       # the same step with forward + backward replayed from a CUDA graph (host-launch bound otherwise)
        loss_fn = lambda: model(srcs, masks, poss, dsrcs, dmasks, dposs, query)[0].float().square().mean()
        graphed = data_parallel.GraphedTrainStep(model, opt, loss_fn)
        ms = _reduce_max(torch, dist, world, dev, _time_events(torch, graphed, iters, 2))
        out["ms_per_step"] = ms
        out["frames_per_s"] = n_frames * world / ms * 1e3
        out["mode"] = "CUDA graph (fwd+bwd) + flat-buffer all-reduce + AdamW"
        same, spread = params_agree()
        out["params_equal_across_ranks_after_graphed_steps"] = same
        out["params_max_spread_after_graphed_steps"] = spread
    except Exception as exc:      # report, do not hide
        out["graph_error"] = repr(exc)[:200]
        out["ms_per_step"], out["frames_per_s"] = out["eager_ms_per_step"], out["eager_frames_per_s"]
    assert out.get("params_equal_across_ranks_after_graphed_steps", True), \
        f"parameters differ across ranks after the graphed data-parallel steps: {out}"
    return out


def run_b200(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from dfvod_b200 import MultiScaleDeformableAttention as MSDA
    from dfvod_b200.host_pipeline import bind_host_thread_near_device
    bound_cores = bind_host_thread_near_device(local)      # pinned buffers below land on the GPU's NUMA node

    tdtype = {"f32": torch.float32, "bf16": torch.bfloat16}[args.dtype]
    e_v = 4 if args.dtype == "f32" else 2
    n = args.batch
    lsi, s = level_start(COCO_SHAPES)
    value_h, loc_h, attn_h, gout_h = make_inputs(torch, n, 1000 + rank, args.dist)
    value_h, gout_h = value_h.to(tdtype), gout_h.to(tdtype)
    host = [t.pin_memory() for t in (value_h, loc_h, attn_h, gout_h)]
    value, loc, attn, gout = (t.to(dev) for t in host)
    st = torch.as_tensor(COCO_SHAPES, dtype=torch.long, device=dev)
    ls = torch.as_tensor(lsi, dtype=torch.long, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_steps(k):
        """k steps, each fwd + bwd through the public boundary; CUDA events around every launch.
        Warm-up and the timed region run this same function, so the caching allocator is in
        steady state (no cudaMalloc inside the timed region)."""
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(k)]
        keep = None
        for i in range(k):
            ev[i][0].record()
            out = MSDA.ms_deform_attn_forward(value, st, ls, loc, attn, 64)
            ev[i][1].record()
            grads = MSDA.ms_deform_attn_backward(value, st, ls, loc, attn, gout, 64)
            ev[i][2].record()
            keep = (out, grads)
        return ev, keep

    run_steps(max(args.warmup, 3))
    barrier()

    # ---- timed region: device-resident inputs ------------------------------------------------
    with ClockSampler(local) as clocks:
        barrier()
        t_start = torch.cuda.Event(enable_timing=True)
        t_end = torch.cuda.Event(enable_timing=True)
        t_start.record()
        ev, last = run_steps(args.steps)
        t_end.record()
        barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, args.dump_outputs, (last[0], *last[1]))
    del last
    elapsed_ms = t_start.elapsed_time(t_end)
    fwd_all = sorted(e[0].elapsed_time(e[1]) for e in ev)
    bwd_all = sorted(e[1].elapsed_time(e[2]) for e in ev)
    fwd_ms, bwd_ms = sum(fwd_all) / args.steps, sum(bwd_all) / args.steps
    fwd_med, bwd_med = fwd_all[len(fwd_all) // 2], bwd_all[len(bwd_all) // 2]
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    total_queries = n * s * world * args.steps
    value_qps = total_queries / (elapsed_ms * 1e-3)

    # ---- end to end: host buffers in, host buffers out, copies inside the timed region ---------
    # the repo's host-buffer entry point (host_pipeline.HostPipelinedMSDA): frames flow through
    # H2D / kernels / D2H on three streams.  Every step moves ALL inputs in and ALL results out.
    from dfvod_b200.host_pipeline import HostPipelinedMSDA
    pinned_out = [torch.empty((n, s, M * D), dtype=tdtype).pin_memory(),
                  torch.empty_like(value_h).pin_memory(), torch.empty_like(loc_h).pin_memory(),
                  torch.empty_like(attn_h).pin_memory()]
    pipe = HostPipelinedMSDA(dev, st.cpu(), ls.cpu(), M, D, P, s, dtype=tdtype, chunk_frames=2, depth=3)

    def e2e_step():
        pipe.forward_backward(*host, *pinned_out)

    e2e_steps = max(2, min(args.steps, 10))
    for _ in range(2):
        e2e_step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(e2e_steps):
        e2e_step()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_qps = n * s * world * e2e_steps / (float(t.item()) * 1e-3)
    h2d = sum(t.numel() * t.element_size() for t in host)
    d2h = sum(t.numel() * t.element_size() for t in pinned_out)
    del pipe

    # ---- what bounds the end-to-end number: the host<->device copy ceiling of this box -----------
    # The same bytes, nothing else: every rank copies its step's inputs in and its results out with plain pinned
    # cudaMemcpyAsync on two streams, all ranks at once (the 8 GPUs of a box share the host's memory system).
    dev_in = [torch.empty_like(t, device=dev) for t in host]
    dev_out = [torch.empty_like(t, device=dev) for t in pinned_out]
    s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def copy_step():
        with torch.cuda.stream(s_in):
            for d_, h_ in zip(dev_in, host):
                d_.copy_(h_, non_blocking=True)
        with torch.cuda.stream(s_out):
            for h_, d_ in zip(pinned_out, dev_out):
                h_.copy_(d_, non_blocking=True)

    copy_step()
    barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    s_in.wait_stream(torch.cuda.current_stream(dev))
    s_out.wait_stream(torch.cuda.current_stream(dev))
    for _ in range(e2e_steps):
        copy_step()
    torch.cuda.current_stream(dev).wait_stream(s_in)
    torch.cuda.current_stream(dev).wait_stream(s_out)
    c1.record()
    barrier()
    t = torch.tensor([c0.elapsed_time(c1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    copy_ms = float(t.item()) / e2e_steps
    copy_limit_qps = n * s * world / (copy_ms * 1e-3)
    e2e_limit = {"value": copy_limit_qps, "unit": UNIT, "ms_per_step": copy_ms,
                 "h2d_gbytes_per_s_all_ranks": h2d * world / copy_ms / 1e6,
                 "d2h_gbytes_per_s_all_ranks": d2h * world / copy_ms / 1e6,
                 "frac_of_limit": e2e_qps / copy_limit_qps,
                 "what": "the step's input and output bytes moved by plain pinned cudaMemcpyAsync on two streams, all "
                         "ranks at once, no kernels: the ceiling of any host-buffer API on this box"}
    del dev_in, dev_out

    # ---- the same end-to-end call with bf16 values / outputs / value gradients (locations, weights fp32) ----------
    e2e_bf16 = None
    if args.dtype == "f32":
        try:
            bft = torch.bfloat16
            host16 = [value_h.to(bft).pin_memory(), loc_h.pin_memory(), attn_h.pin_memory(), gout_h.to(bft).pin_memory()]
            out16 = [torch.empty((n, s, M * D), dtype=bft).pin_memory(), torch.empty(value_h.shape, dtype=bft).pin_memory(),
                     torch.empty_like(loc_h).pin_memory(), torch.empty_like(attn_h).pin_memory()]
            pipe16 = HostPipelinedMSDA(dev, st.cpu(), ls.cpu(), M, D, P, s, dtype=bft, chunk_frames=2, depth=3)
            for _ in range(2):
                pipe16.forward_backward(*host16, *out16)
            barrier()
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0.record()
            for _ in range(e2e_steps):
                pipe16.forward_backward(*host16, *out16)
            b1.record()
            barrier()
            t = torch.tensor([b0.elapsed_time(b1)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            h16 = sum(x.numel() * x.element_size() for x in host16)
            d16 = sum(x.numel() * x.element_size() for x in out16)
            q16 = n * s * world * e2e_steps / (float(t.item()) * 1e-3)
            # the copy ceiling scales with the bytes: the measured fp32 ceiling (bytes per second) applied to these bytes
            lim16 = copy_limit_qps * (h2d + d2h) / (h16 + d16)
            e2e_bf16 = {"value": q16, "unit": UNIT, "h2d_bytes_per_step": h16, "d2h_bytes_per_step": d16,
                        "steps": e2e_steps, "limit_from_measured_copy_rate": lim16, "frac_of_limit": q16 / lim16}
            del pipe16, host16, out16
        except Exception as exc:
            e2e_bf16 = {"error": repr(exc)[:200]}

    # ---- the other storage type of the op (bf16 values when the line is fp32 and vice versa): device-resident --
    other = {}
    try:
        odt, oname, oe = (torch.bfloat16, "bf16", 2) if args.dtype == "f32" else (torch.float32, "f32", 4)
        v2, g2 = value.to(odt), gout.to(odt)
        f_ms = _time_events(torch, lambda: MSDA.ms_deform_attn_forward(v2, st, ls, loc, attn, 64), 10, 3)
        b_ms = _time_events(torch, lambda: MSDA.ms_deform_attn_backward(v2, st, ls, loc, attn, g2, 64), 10, 3)
        f_ms = _reduce_max(torch, dist, world, dev, f_ms)
        b_ms = _reduce_max(torch, dist, world, dev, b_ms)
        fb, bb = algorithmic_bytes(n, oe)
        pk, _ = peaks()
        other = {"dtype": oname, "fwd_ms": f_ms, "bwd_ms": b_ms, "value": n * s * world / ((f_ms + b_ms) * 1e-3),
                 "unit": UNIT, "roofline_frac_fwd": fb / (f_ms * 1e-3) / 1e9 / pk,
                 "roofline_frac_bwd": bb / (b_ms * 1e-3) / 1e9 / pk}
        del v2, g2
    except Exception as exc:
        other = {"error": repr(exc)[:200]}

    # ---- roofline of the dominant kernel (the backward) ----------------------------------------
    peak, peak_src = peaks()
    fwd_bytes, bwd_bytes = algorithmic_bytes(n, e_v)
    achieved_bwd = bwd_bytes / (bwd_ms * 1e-3) / 1e9
    achieved_fwd = fwd_bytes / (fwd_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "msda_bwd_fast_kernel (+ its grad_value zero-fill"
                                          + (" and bf16 cast" if e_v == 2 else "") + ")",
                "achieved": achieved_bwd, "peak": peak, "unit": "GB/s", "frac": achieved_bwd / peak,
                "traffic": traffic_from_profile("backward", args.dtype), "peak_source": peak_src,
                "traffic_capture_is_of_this_build": profile_build_matches(),
                "algorithmic_bytes_per_launch": bwd_bytes, "ms_per_launch": bwd_ms,
                "limiter": limiter_from_profile("backward", args.dtype)}
    roofline_fwd = {"bound": "hbm", "kernel": "msda_fwd_fast_kernel", "achieved": achieved_fwd, "peak": peak,
                    "unit": "GB/s", "frac": achieved_fwd / peak, "traffic": traffic_from_profile("forward", args.dtype),
                    "algorithmic_bytes_per_launch": fwd_bytes, "ms_per_launch": fwd_ms,
                    "limiter": limiter_from_profile("forward", args.dtype)}

    extras = {}
    if not args.no_extras:
        del value, loc, attn, gout, host, pinned_out          # give the memory back first
        torch.cuda.empty_cache()
        for name, fn in (("detr_inference", encoder_extras), ("encoder_cross_fusion_layer", fusion_layer_extras),
                         ("transvod_clip_inference", clip_extras), ("input_projections", input_projection_extras),
                         ("train_step", train_step_extras)):
            try:
                extras[name] = fn(torch, dev, world, dist)
            except Exception as exc:                          # extras never invalidate the main line
                extras[name] = {"error": repr(exc)[:200]}
            torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        cb = time_cpu_reference(torch, 30, 1, args.dist)          # ~10 s of host work
        cpu_baseline = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}

    line = {"metric": METRIC, "value": value_qps, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": "msda_core_op_fwd_bwd_coco_pyramid_800x1333", "levels": COCO_SHAPES,
                       "queries_per_frame": s, "heads": M, "head_dim": D, "points": P,
                       "frames_per_step_per_gpu": n, "loc_distribution": args.dist,
                       "l2": "inputs (%d MB per step) larger than L2" % ((fwd_bytes + bwd_bytes) // (2 << 20)),
                       "parallelism": f"dp{world} (frames sharded, no data-path collective)"},
            "e2e": {"value": e2e_qps, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "host_cores_bound_near_gpu": bound_cores, "limit": e2e_limit,
                    "api": "dfvod_b200.host_pipeline.HostPipelinedMSDA.forward_backward (pinned host tensors)"},
            "gpu_launches": args.steps * (2 if e_v == 4 else 3),
            "clocks": clocks.summary(),
            "roofline": roofline, "roofline_fwd": roofline_fwd,
            "fwd_ms": fwd_ms, "bwd_ms": bwd_ms,
            "per_step_ms": {"fwd_median": fwd_med, "bwd_median": bwd_med, "fwd_min": fwd_all[0],
                            "bwd_min": bwd_all[0], "fwd_max": fwd_all[-1], "bwd_max": bwd_all[-1]},
            "op_other_dtype": other, "e2e_bf16": e2e_bf16,
            "cpu_baseline": cpu_baseline}
    line.update(extras)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dtype", default="f32", choices=["f32", "bf16"])
    ap.add_argument("--dist", default="grid", choices=["grid", "random", "init"])
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the encoder / training-step side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the op's results of the last timed step as DIR/<name>.npy (float32, <= 64 MiB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
