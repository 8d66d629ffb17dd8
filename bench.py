#!/usr/bin/env python
"""bench.py — fwd+bwd ms/view of SplatCo's differentiable render hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2] [--dump-outputs DIR]

A "step" is one training iteration's render work for the `--mv` multi-view batch (BASELINE.json
configs[1]: Tanks&Temples-shaped, 100k anchors x 10 offsets ~ 1M candidate Gaussians, 980x545, mv=4):
for every view   prefilter_voxel -> generate_neural_gaussians (fused decode) -> preprocess ->
binning/sort -> blend,   the reference's per-view loss terms that touch the hot path's outputs
(0.8*L1 + 0.2*(1-SSIM) + 0.01*mean(prod(scaling)), train.py:192-196; the image part is the fused
l1_ssim_loss of SURVEY §8 row f3),   then ONE
backward over the summed loss (train.py:240), through the drop-in `gaussian_renderer.render()`.
With N > 1 every rank renders its own mv views (weak scaling, views sharded by rank) and the
parameter gradients are all-reduced with NCCL.

Printed JSON (one line, rank 0): metric fwd_bwd_ms_per_view (lower is better) = max-over-ranks step
time / views rendered by all ranks, inputs resident in HBM; `e2e` = the same with host inputs (each
view's ground-truth image copied H2D from pinned memory, the loss read back D2H every step);
`roofline` for the stage with the largest share (with the blend's issue-slot roofline: live (pixel, instance) pairs,
warp instructions per live pair); `decode_mlp` = the tcgen05 MLP kernels timed with CUDA events in this run;
`cpu_baseline` = the oracle port on the host cores over one view; `parity` = this run's view 0 (Q0 = 0) against that
oracle rendering; `gpu_baseline` = same-GPU comparators (torch-eager decode, upstream-structure rasterizer);
`sub_records` = BASELINE configs[2] (C3) at one GPU / configs[3] (C4, one view per GPU) at eight, measured the same way;
`multi_gpu_check` (N > 1) = one checked step of the view-sharded path on NCCL against a single-process evaluation.

`--dump-outputs DIR` (rank 0): what the last step of the timed loop computed -- every view's rendered image, the summed
loss and every parameter gradient -- as DIR/<name>.npy in float32, so that two builds can be compared output for
output (the inputs of the timed steps depend only on the arguments).  Arrays larger than DUMP_MAX_ELEMS are stored as
the same seeded sample of their entries in every run.

`--impl reference`: the reference's rasterizer is CUDA-only and absent from the mount and its Python
decode cannot travel to the GPU box (SURVEY.md §0.1, §8c), so this arm times the oracle port of the
same path (oracle/decode_oracle.py on torch CPU threads + oracle/raster_oracle.c on all host
threads), one view of the workload per step.
"""
from __future__ import annotations

import argparse
import gc
import json
import math
import os
import subprocess
import sys
import tempfile
import time
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

WORKLOADS = {
    "c1": dict(N=10_000, K=10, W=256, H=256, mv=1, plane_size=512, C=15,
               desc="C1 synthetic 10k anchors x10 offsets, 256x256, 1 view"),
    "c2": dict(N=100_000, K=10, W=980, H=545, mv=4, plane_size=2500, C=15,
               desc="C2 Tanks&Temples-shaped 100k anchors x10 offsets (~1M Gaussians), 980x545, mv=4"),
    "c3": dict(N=500_000, K=10, W=1152, H=864, mv=4, plane_size=2800, C=15,
               desc="C3 Mill19-Rubble-shaped 500k anchors x10 (~5M Gaussians), 1152x864, plane_size 2800, mv=4"),
    "c4": dict(N=1_000_000, K=10, W=1920, H=1080, mv=1, plane_size=2800, C=15,
               desc="C4 MatrixCity-Aerial-shaped 1M anchors x10 (~10M Gaussians), 1920x1080, one view per GPU (mv=8 over 8 GPUs)"),
}
SCALE_FACTOR = 0.5       # anchor scale = 0.5 / N^(1/3): projected sigma ~0.5-4 px at these resolutions (SURVEY §8d)
LEVEL = 2                # activate_level in steady state (train.py:305-307)
DUMP_MAX_ELEMS = 1 << 19  # --dump-outputs: 2 MB per array; C2 and C3 reach it with 16 arrays (4 images, 12 gradients), ~33 MB
DUMP_MAX_BYTES = 64 << 20


def ncu_evidence():
    """Per-kernel numbers of the latest committed `ncu --set full` capture (profiles/*_traffic.json, written by
    tools/collect_profiles.py): dram bytes per launch, issue-active, tensor-pipe-active."""
    d = os.path.join(ROOT, "profiles")
    # capture tags grow r1a .. r1z, r2a .. r2z, r2aa ..: order by (length, name)
    files = sorted((f for f in os.listdir(d) if f.endswith("_traffic.json")), key=lambda f: (len(f), f)) if os.path.isdir(d) else []
    if not files:
        return {}
    ev = json.load(open(os.path.join(d, files[-1])))
    ev["_file"] = "profiles/" + files[-1]
    return ev


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        if os.environ.get("SPLATCO_BENCH_NO_SAMPLER") == "1":       # diagnostic: is the poller itself disturbing the run?
            return
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        try:
            rows = [r.split(",") for r in open(self.path).read().strip().splitlines() if r.strip()]
            rows = [r for r in rows if len(r) >= 9]
            if rows:
                out["sm_mhz"] = float(np.median([float(r[1]) for r in rows]))
                out["sm_max_mhz"] = float(rows[0][2])
                out["power_w_max"] = max(float(r[3]) for r in rows)
                for k, n in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
                    if any(r[5 + k].strip() == "Active" for r in rows):
                        out["reasons"].append(n)
                out["samples"] = len(rows)
            os.unlink(self.path)
        except Exception:
            pass
        return out


def build_model(cfg, device, seed=1):
    from splatco_b200.model import AnchorModel
    pc = AnchorModel(cfg["N"], n_offsets=cfg["K"], plane_size=cfg["plane_size"], num_channels=cfg["C"],
                     device=device, seed=20240 + seed, scale_factor=SCALE_FACTOR)
    pc.feat_planes._feat.activate_level = LEVEL
    pc.train()
    return pc


def build_views(cfg, rank=0, world=1, seed=1):
    from splatco_b200.synthetic import ring_cameras
    phase = 2 * math.pi * rank / (world * cfg["mv"]) if world > 1 else 0.0
    cams = ring_cameras(cfg["mv"], cfg["W"], cfg["H"], phase=phase)
    g = torch.Generator().manual_seed(777 + seed + rank)
    gts = [torch.rand(3, cfg["H"], cfg["W"], generator=g) for _ in cams]
    return cams, gts


PIPE = SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False)


def _tf32_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["bf16_tflops"] / 2, "measured (half of the bf16 cuBLAS burst figure)"
    return 795.0, "fallback (half of 1.59 PFLOP/s)"


class Workload:
    """One configuration resident on this rank's GPU: model, cameras, ground truth (device + pinned host), step()."""

    def __init__(self, args, name, device, rank, world):
        from splatco_b200.multiview import GradBucket
        self.args, self.name, self.device, self.rank, self.world = args, name, device, rank, world
        self.cfg = cfg = WORKLOADS[name]
        self.pc = build_model(cfg, device)
        self.pc.feat_planes.Q0 = 0.03                      # training-time plane-feature noise (timing config, SURVEY §8d)
        cams, gts = build_views(cfg, rank, world)
        self.cams = [c.to(device) for c in cams]
        self.bg = torch.ones(3, device=device)
        self.gts_dev = [g.to(device) for g in gts]
        self.gts_pinned = [g.pin_memory() for g in gts]
        self.params = self.pc.parameters()
        self.bucket = GradBucket(self.params) if world > 1 else None
        self.mv = cfg["mv"]
        # e2e: each step's ground-truth images leave pinned host memory inside the timed region, on a copy stream into
        # fixed staging buffers (what a data loader does); a view waits for its own image only when it computes its loss
        self.copy_stream = torch.cuda.Stream(device)
        self.gts_stage = [torch.empty_like(g) for g in self.gts_dev]
        self.copied = [torch.cuda.Event() for _ in range(self.mv)]
        self.info = {}
        self.host_ms = {}
        self.keep_outputs = False       # --dump-outputs: step() keeps its rendered images and loss in self.last
        self.last = None

    def step(self, host_inputs: bool):
        from splatco_b200.gaussian_renderer import prefilter_voxel, render
        from splatco_b200.loss import l1_ssim_loss, scaling_reg
        a, device, mv = self.args, self.device, self.mv
        for p in self.params:
            p.grad = None
        self.last = None                # (released before this step allocates its own)
        total = None
        Ms, Vs, renders = [], [], []
        if host_inputs:
            self.copy_stream.wait_stream(torch.cuda.current_stream(device))     # the previous step no longer reads the buffers
            with torch.cuda.stream(self.copy_stream):
                for v in range(mv):
                    self.gts_stage[v].copy_(self.gts_pinned[v], non_blocking=True)
                    self.copied[v].record(self.copy_stream)
        for v in range(mv):
            vm = prefilter_voxel(self.cams[v], self.pc, PIPE, self.bg)
            pkg = render(self.cams[v], self.pc, PIPE, self.bg, visible_mask=vm, retain_grad=True)
            if host_inputs:
                torch.cuda.current_stream(device).wait_event(self.copied[v])
                gt = self.gts_stage[v]
            else:
                gt = self.gts_dev[v]
            # the reference's per-view loss (train.py:192-196, lambda_dssim = 0.2 from arguments/__init__.py), image part fused
            loss = l1_ssim_loss(pkg["render"], gt, 0.2) + 0.01 * (pkg["scaling"].prod(dim=1).mean() if a.torch_scaling_reg else scaling_reg(pkg["scaling"]))
            total = loss if total is None else total + loss
            Ms.append(pkg["radii"].shape[0]); Vs.append(pkg["selection_mask"].shape[0] // self.cfg["K"])
            if self.keep_outputs:
                renders.append(pkg["render"].detach())
        total.backward()
        if self.bucket is not None:
            self.bucket.allreduce()
        if self.keep_outputs:
            self.last = (renders, total.detach())
        self.info["M"], self.info["V"] = float(np.mean(Ms)), float(np.mean(Vs))
        return float(total.item()) if host_inputs else total

    def outputs(self):
        """Host copies (dump_sample) of what the last step() handed its caller: the rendered image of every view, the
        summed loss and the gradient of every parameter (None gradients left out), keyed by the names --dump-outputs
        writes."""
        renders, loss = self.last
        out = {f"render_view{v}": r for v, r in enumerate(renders)}
        out["loss"] = loss
        pc = self.pc
        named = {k: getattr(pc, k) for k in ("_anchor", "_offset", "_anchor_feat", "_scaling")}
        for m in ("mlp_opacity", "mlp_cov", "mlp_color", "feat_planes"):
            named.update({f"{m}.{k}": p for k, p in getattr(pc, m).named_parameters()})
        out.update({f"grad.{k}": p.grad for k, p in named.items() if p.grad is not None})
        return {k: dump_sample(t.cpu().numpy()) for k, t in out.items()}

    def timed(self, fn, n, host_inputs, tag=None):
        import torch.distributed as dist
        # the cyclic collector is paused inside the timed region (a generation-2 pass over the autograd graphs of a
        # step costs tens of ms and lands on a random step); per-step host times are kept as a diagnostic
        gc.collect()
        gc.disable()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ts = [time.perf_counter()]
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(n)]
        st0 = torch.cuda.memory_stats(self.device)
        memhist = os.environ.get("SPLATCO_BENCH_MEMHIST") == "1"        # diagnostic: who asks for new segments in here?
        if memhist:
            torch.cuda.memory._record_memory_history(max_entries=200000)
        e0.record()
        for i in range(n):
            fn(host_inputs)
            marks[i].record()
            ts.append(time.perf_counter())
        e1.record()
        torch.cuda.synchronize()
        gc.enable()
        st1 = torch.cuda.memory_stats(self.device)
        if memhist:
            snap = torch.cuda.memory._snapshot()
            torch.cuda.memory._record_memory_history(enabled=None)
            seen = []
            for tr in snap.get("device_traces", []):
                for k, ev in enumerate(tr):
                    if ev.get("action") == "segment_alloc":
                        # the allocation request that follows the new segment carries the Python stack
                        nxt = next((e for e in tr[k + 1:k + 4] if e.get("action") == "alloc"), ev)
                        fr = [f"{os.path.basename(f['filename'])}:{f['line']}:{f['name']}" for f in nxt.get("frames", []) if f["filename"].endswith(".py") and "site-packages" not in f["filename"]][:8]
                        seen.append({"size_mb": round(ev["size"] / 1e6, 1), "frames": fr})
            sys.stderr.write(f"[memhist rank {self.rank} {tag or getattr(fn, '__name__', 'fn')}] " + json.dumps(seen) + "\n")
        d = sorted((b - a) * 1e3 for a, b in zip(ts[:-1], ts[1:]))
        gd = sorted(a.elapsed_time(b) for a, b in zip([e0] + marks[:-1], marks))
        tag = tag or (getattr(fn, "__name__", "fn") + ("_host_inputs" if host_inputs else ""))
        self.host_ms[tag] = {
            "host_median": round(d[len(d) // 2], 3), "host_max": round(d[-1], 3),
            "gpu_median": round(gd[len(gd) // 2], 3), "gpu_max": round(gd[-1], 3),
            # cudaMalloc / cudaFree calls of torch's caching allocator inside the timed region (0 / 0 in steady state)
            "cuda_mallocs": int(st1.get("num_device_alloc", 0) - st0.get("num_device_alloc", 0)),
            "cuda_frees": int(st1.get("num_device_free", 0) - st0.get("num_device_free", 0)),
            "reserved_mb_grown": {k: round((st1.get(f"reserved_bytes.{k}.current", 0) - st0.get(f"reserved_bytes.{k}.current", 0)) / 1e6, 1)
                                  for k in ("large_pool", "small_pool")}}
        if self.world > 1:
            dist.barrier()
        ms = e0.elapsed_time(e1)
        if self.world > 1:
            # diagnostic: every rank's own total and slowest step (the reported time is the max over ranks)
            mine = torch.tensor([ms, gd[-1], gd[len(gd) // 2], float(self.host_ms[tag]["cuda_mallocs"])], device=self.device)
            allr = [torch.zeros_like(mine) for _ in range(self.world)]
            dist.all_gather(allr, mine)
            self.host_ms[tag]["per_rank"] = [
                {"total_ms": round(float(a[0]), 2), "gpu_max": round(float(a[1]), 2), "gpu_median": round(float(a[2]), 2),
                 "cuda_mallocs": int(a[3])} for a in allr]
            ms = max(float(a[0]) for a in allr)
        return ms

    def instance_counts(self):
        """Instance count R and the blend's work census (visited / live (pixel, instance) pairs) of each view."""
        from splatco_b200 import _lib
        from splatco_b200._lib import check, ptr
        from splatco_b200.diff_gaussian_rasterization import rasterize_forward_state
        from splatco_b200.gaussian_renderer import _settings, generate_neural_gaussians, prefilter_voxel
        L = _lib.lib()
        H, W = self.cfg["H"], self.cfg["W"]
        Rs, visited, live = [], [], []
        out = torch.zeros(2, dtype=torch.int64, device=self.device)
        with torch.no_grad():
            for v in range(self.mv):
                vm = prefilter_voxel(self.cams[v], self.pc, PIPE, self.bg)
                xyz, color, opacity, scaling, rot, _, _ = generate_neural_gaussians(self.cams[v], self.pc, vm, is_training=True)
                _, _, st = rasterize_forward_state(xyz, color, opacity, scaling, rot, _settings(self.cams[v], PIPE, self.bg, 1.0))
                Rs.append(st.R)
                if st.R > 0:
                    check(L.splatco_blend_census(st.RL, H, W, ptr(st.geom), ptr(st.binning), ptr(st.image), ptr(out),
                                                 _lib.raw_stream(self.device)), "splatco_blend_census")
                    o = out.cpu().numpy()
                    visited.append(int(o[0])); live.append(int(o[1]))
        return float(np.mean(Rs)), float(np.mean(visited or [0])), float(np.mean(live or [0]))


def dump_sample(a):
    """`a` as float32; an array of more than DUMP_MAX_ELEMS entries becomes its entries at DUMP_MAX_ELEMS positions
    drawn (seed 0, sorted) from its flattened shape, the same positions in every run."""
    a = np.asarray(a, np.float32)
    if a.size > DUMP_MAX_ELEMS:
        idx = np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))
        a = a.reshape(-1)[idx]
    return a


def dump_outputs(d, arrays):
    """Writes d/<name>.npy (float32) for every array, or nothing if they add up to more than DUMP_MAX_BYTES."""
    arrays = {k: np.asarray(a, np.float32) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total / 2**20:.1f} MB is more than {DUMP_MAX_BYTES >> 20} MB")
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), a)


def stage_table(w: Workload, stage_sum, ms_stage, R, M, V):
    cfg = w.cfg
    N, H, W = cfg["N"], cfg["H"], cfg["W"]
    HW = H * W
    T = ((W + 15) // 16) * ((H + 15) // 16)
    passes = math.ceil((32 + max(1, (T - 1).bit_length())) / 8)
    dec_bytes = V * (284 + 240 * (LEVEL + 2) + 50) + 56 * M          # SURVEY §8d decode fwd per visible anchor
    alg_bytes = {                                                      # SURVEY §8d / BASELINE.md §3.4
        "visible_filter": 48.0 * N,
        "decode_fwd": dec_bytes, "decode_emit": 56.0 * M, "decode_bwd": 2.0 * dec_bytes,
        "preprocess_fwd": 104.0 * M,
        "binning": 12.0 * R + passes * 24.0 * R + 8.0 * R + 8.0 * R + 8.0 * T,
        "blend_fwd": 40.0 * R + 20.0 * HW,
        "blend_bwd": 76.0 * R + 32.0 * HW,
        "preprocess_bwd": 200.0 * M,
    }
    stages = {}
    for k, (n, tot) in stage_sum.items():
        avg = tot / max(n, 1)
        st = {"calls": n, "avg_ms": round(avg, 4), "share": round(tot / ms_stage, 4)}
        if k in alg_bytes and avg > 0:
            st["alg_gbs"] = round(alg_bytes[k] / (avg * 1e-3) / 1e9, 1)
        stages[k] = st
    timed_k = [k for k in stage_sum if k in alg_bytes]
    dom = max(timed_k, key=lambda k: stage_sum[k][1]) if timed_k else None
    return stages, alg_bytes, dom


def warm_until_quiescent(w, device, world, limit=24, batch=4):
    """Extra untimed steps, in free-running batches like the timed loop (how many gradient arenas c10d still holds -- and so
    how far the arena pool has to grow -- depends on how fast the host issues steps), until a batch passes without a
    cudaMalloc of torch's caching allocator on any rank; returns how many steps were run."""
    import torch.distributed as dist
    extra = 0
    while extra < limit:
        n0 = torch.cuda.memory_stats(device).get("num_device_alloc", 0)
        for _ in range(batch):
            w.step(False)
        extra += batch
        torch.cuda.synchronize()
        grew = torch.tensor([float(torch.cuda.memory_stats(device).get("num_device_alloc", 0) - n0)], device=device)
        if world > 1:
            dist.all_reduce(grew, op=dist.ReduceOp.MAX)
        if float(grew.item()) == 0.0:
            break
    return extra


def sub_record(args, name, device, rank, world, warm=3):
    """A measurement of another BASELINE config inside the same bench line (--steps timed steps): value, e2e,
    dominant-stage roofline."""
    from splatco_b200 import profiling
    steps = args.steps
    w = Workload(args, name, device, rank, world)
    for _ in range(warm):
        w.step(False)
    warm += warm_until_quiescent(w, device, world, limit=8, batch=4)
    ms_dev = w.timed(w.step, steps, False)
    ms_e2e = w.timed(w.step, steps, True)
    with profiling.collect() as prof:
        ms_stage = w.timed(w.step, steps, False)
    rec = None
    if rank == 0:
        R, _, _ = w.instance_counts()
        stages, alg_bytes, dom = stage_table(w, prof.summary(), ms_stage, R, w.info["M"], w.info["V"])
        peak, peak_src = peaks()
        views = w.mv * world
        rec = {"workload": w.cfg["desc"], "value": round(ms_dev / steps / views, 4), "unit": "ms/view", "ms_per_step": round(ms_dev / steps, 4),
               "steps": steps, "warmup": warm, "n_gpus": world, "views_per_step": views,
               "e2e": {"value": round(ms_e2e / steps / views, 4), "unit": "ms/view"},
               "visible_anchors": int(w.info["V"]), "gaussians": int(w.info["M"]), "instances_R": int(R),
               "stages_ms": {k: v["avg_ms"] for k, v in stages.items()}}
        if dom:
            rec["roofline"] = {"kernel": dom, "bound": "hbm", "achieved": stages[dom]["alg_gbs"], "peak": peak, "unit": "GB/s",
                               "frac": round(stages[dom]["alg_gbs"] / peak, 4), "peak_source": peak_src,
                               "alg_bytes_per_launch": int(alg_bytes[dom])}
        if w.bucket is not None:
            rec["allreduce_bytes_per_step"] = w.bucket.nbytes()
    del w
    gc.collect()
    torch.cuda.empty_cache()
    return rec


def gpu_baseline(w: Workload):
    """Same-GPU comparators (BASELINE.md §3.2; the reference's CUDA rasterizer is absent from the mount):
      decode: the reference's PyTorch decode on this B200 -- its OWN generate_neural_gaussians + FeaturePlanes when
              oracle/_ref is staged (oracle/build_ref.py), else the plain-torch restatement oracle/decode_oracle.py on cuda;
      rasterizer: the upstream STRUCTURE restated (csrc/blend_upstream.cu: 256-instance batches, every pixel evaluates
              every instance, per-pixel atomics) behind the literal duplicateWithKeys + 6-pass radix + identifyTileRanges
              composition, on the same Gaussians, against the product kernels on the same workspaces."""
    from splatco_b200 import _lib
    from splatco_b200._lib import check, ptr
    from splatco_b200.diff_gaussian_rasterization import rasterize_forward_state
    from splatco_b200.gaussian_renderer import _settings, generate_neural_gaussians, prefilter_voxel
    L = _lib.lib()
    dev, cfg, pc = w.device, w.cfg, w.pc
    H, W = cfg["H"], cfg["W"]
    cam = w.cams[0]
    out = {}

    def time_ms(fn, n=5, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    q0 = pc.feat_planes.Q0
    with torch.no_grad():
        vm = prefilter_voxel(cam, pc, PIPE, w.bg)
    # ---- decode: torch eager on the same GPU ----
    try:
        from oracle import decode_oracle as D
        p = {"feat." + k: v for k, v in pc.feat_planes._feat.state_dict().items()}
        for name in ("mlp_opacity", "mlp_cov", "mlp_color"):
            p.update({f"{name}.{k}": v for k, v in getattr(pc, name).state_dict().items()})
        p = {k: (v.detach().clone().requires_grad_(True) if v.dtype.is_floating_point and "running" not in k and "xyz_m" not in k else v)
             for k, v in p.items()}
        leaves = [t.detach().clone().requires_grad_(True) for t in (pc._anchor_feat, pc._anchor, pc._offset, pc._scaling)]

        def torch_decode():
            for t in leaves + [v for v in p.values() if v.requires_grad]:
                t.grad = None
            outs = D.decode(p, leaves[0], leaves[1], leaves[2], torch.exp(leaves[3]), vm, cam.camera_center, LEVEL, cfg["K"])
            sum((o.sum() for o in outs[:5])).backward()

        def ours_decode():
            for t in w.params:
                t.grad = None
            outs = generate_neural_gaussians(cam, pc, vm, is_training=True)
            sum((o.sum() for o in outs[:5])).backward()

        pc.feat_planes.Q0 = 0.0
        t_torch = time_ms(torch_decode, n=3, warm=1)
        t_ours = time_ms(ours_decode, n=5, warm=2)
        out["decode_fwd_bwd"] = {"torch_eager_ms": round(t_torch, 3), "ours_ms": round(t_ours, 3), "ratio": round(t_torch / t_ours, 2),
                                 "kind": "port", "what": "oracle/decode_oracle.py (plain-torch restatement of generate_neural_gaussians + "
                                 "FeaturePlanes, pinned to the reference's fixtures) on the same B200, one view, fwd + autograd bwd; ours = "
                                 "generate_neural_gaussians through the C ABI incl. its host side"}
    except Exception as e:      # the comparator must never take the bench line down
        out["decode_fwd_bwd"] = {"error": repr(e)[:200]}
    finally:
        pc.feat_planes.Q0 = q0
    # ---- rasterizer: upstream structure on the same Gaussians / workspaces ----
    try:
        with torch.no_grad():
            xyz, color, opacity, scaling, rot, _, _ = generate_neural_gaussians(cam, pc, vm, is_training=True)
            settings = _settings(cam, PIPE, w.bg, 1.0)
            img, radii, st = rasterize_forward_state(xyz, color, opacity, scaling, rot, settings)
        stream = _lib.raw_stream(dev)
        P, R = st.P, st.R
        bin2 = torch.empty_like(st.binning)
        img2 = torch.empty_like(st.image)
        col2 = torch.empty_like(img)
        dL = torch.randn_like(img) * 1e-3
        g = [torch.zeros(P, c, device=dev) for c in (3, 3, 1, 3)]

        def zero():
            for t in g:
                t.zero_()

        def up_bin():
            check(L.splatco_binning_radix(st.PL, R, H, W, ptr(st.radii_full), ptr(st.geom), ptr(bin2), ptr(img2), stream), "binning_radix")

        def our_bin():
            check(L.splatco_binning(st.PL, R, H, W, ptr(st.radii_full), ptr(st.geom), ptr(bin2), ptr(img2), stream), "binning")

        def up_fwd():
            check(L.splatco_blend_fwd_upstream(R, H, W, ptr(w.bg), ptr(st.geom), ptr(bin2), ptr(img2), ptr(col2), stream), "blend_fwd_upstream")

        def our_fwd():
            check(L.splatco_blend_fwd(R, H, W, ptr(w.bg), ptr(st.geom), ptr(bin2), ptr(img2), ptr(col2), stream), "blend_fwd")

        def up_bwd():
            zero()
            check(L.splatco_blend_bwd_upstream(P, R, H, W, ptr(w.bg), ptr(st.geom), ptr(bin2), ptr(img2), ptr(dL), *[ptr(t) for t in g], stream),
                  "blend_bwd_upstream")

        def our_bwd():
            zero()
            check(L.splatco_blend_bwd(P, R, H, W, ptr(w.bg), ptr(st.geom), ptr(bin2), ptr(img2), ptr(dL), *[ptr(t) for t in g], stream), "blend_bwd")

        t_zero = time_ms(zero)
        res = {}
        res["binning_upstream_ms"] = round(time_ms(up_bin), 4)
        res["blend_fwd_upstream_ms"] = round(time_ms(up_fwd), 4)
        res["blend_bwd_upstream_ms"] = round(time_ms(up_bwd) - t_zero, 4)
        res["binning_ours_ms"] = round(time_ms(our_bin), 4)          # (also restores the tile order the product blend launches by)
        res["blend_fwd_ours_ms"] = round(time_ms(our_fwd), 4)
        res["blend_bwd_ours_ms"] = round(time_ms(our_bwd) - t_zero, 4)
        up = res["binning_upstream_ms"] + res["blend_fwd_upstream_ms"] + res["blend_bwd_upstream_ms"]
        our = res["binning_ours_ms"] + res["blend_fwd_ours_ms"] + res["blend_bwd_ours_ms"]
        res.update({"upstream_total_ms": round(up, 4), "ours_total_ms": round(our, 4), "ratio": round(up / our, 2), "gaussians": int(P), "instances_R": int(R),
                    "what": "restated upstream, builder-authored (the reference's CUDA source is absent): literal duplicateWithKeys + "
                            "radix sort + identifyTileRanges, 256-batch blend forward, per-pixel-atomic blend backward; same inputs, one view"})
        out["rasterizer_upstream_structure"] = res
    except Exception as e:
        out["rasterizer_upstream_structure"] = {"error": repr(e)[:200]}
    return out


def multi_gpu_check(w: Workload):
    """One CHECKED step of the view-sharded path on real NCCL (not timed): `world` views, one per rank, with the
    cross-view consistency term (all_gather of the rendered images), gradient all-reduce, last-view statistics
    broadcast and an integer count all-reduce; rank 0 then renders all views alone and compares."""
    import torch.distributed as dist
    from splatco_b200.gaussian_renderer import prefilter_voxel, render
    from splatco_b200.loss import l1_ssim_loss, multiview_consistency_loss
    from splatco_b200.multiview import (allreduce_count, broadcast_last_view_stats, shard_views, sharded_consistency_loss)
    from splatco_b200.synthetic import ring_cameras
    world, rank, dev, cfg, pc = w.world, w.rank, w.device, w.cfg, w.pc
    nv = world
    cams = [c.to(dev) for c in ring_cameras(nv, cfg["W"], cfg["H"])]
    g = torch.Generator().manual_seed(4242)
    base = torch.rand(3, cfg["H"], cfg["W"], generator=g)
    reals = [(base + 0.02 * torch.randn(3, cfg["H"], cfg["W"], generator=g)).clamp(0, 1).to(dev) for _ in range(nv)]
    q0 = pc.feat_planes.Q0
    pc.feat_planes.Q0 = 0.0
    if not hasattr(pc, "opacity_accum") or pc.opacity_accum is None or pc.opacity_accum.numel() == 0:
        pc.training_setup()
    stats = [pc.opacity_accum, pc.anchor_demon, pc.offset_gradient_accum, pc.offset_denom]

    def run(views, sharded):
        for p in w.params:
            p.grad = None
        for t in stats:
            t.zero_()
        gens, total, last = [], None, None
        for i in views:
            vm = prefilter_voxel(cams[i], pc, PIPE, w.bg)
            pkg = render(cams[i], pc, PIPE, w.bg, visible_mask=vm, retain_grad=True)
            gens.append(pkg["render"])
            loss = l1_ssim_loss(pkg["render"], reals[i], 0.2)
            total = loss if total is None else total + loss
            if i == nv - 1:
                last = (pkg, vm)
        if sharded:
            total = total + sharded_consistency_loss(gens, reals, nv, rank, world)
        else:
            total = total + multiview_consistency_loss(gens, reals)
        total.backward()
        if sharded:
            w.bucket.allreduce()
        nvis = 0
        if last is not None:          # training_statis consumes the LAST view's tensors only (train.py:266)
            pkg, vm = last
            pc.training_statis(pkg["viewspace_points"], pkg["neural_opacity"], pkg["visibility_filter"], pkg["selection_mask"], vm)
            nvis = int(pkg["visibility_filter"].sum().item())
        if sharded:
            broadcast_last_view_stats(stats, nv)
            nvis = allreduce_count(nvis, dev)
        return [None if p.grad is None else p.grad.detach().clone() for p in w.params], [t.clone() for t in stats], nvis

    got_g, got_s, got_n = run(shard_views(nv, rank, world), True)
    res = None
    if rank == 0:
        want_g, want_s, want_n = run(range(nv), False)
        worst = 0.0
        for a, b in zip(got_g, want_g):
            if a is None or b is None:
                if (a is None) != (b is None):
                    worst = float("inf")
                continue
            scale = max(float(b.abs().max()), 1e-20)
            worst = max(worst, float((a - b).abs().max()) / scale)
        # counters (anchor_demon, offset_denom: integer-valued) must be identical; the two sums of floats (opacity, screen-space
        # gradient norms) come from kernels whose atomics reorder fp32 additions from run to run: 1e-4 of their largest entry
        counters_equal = bool(torch.equal(got_s[1], want_s[1]) and torch.equal(got_s[3], want_s[3]))
        sums_close = bool(all(float((a - b).abs().max()) <= 1e-4 * max(float(b.abs().max()), 1e-20) for a, b in ((got_s[0], want_s[0]), (got_s[2], want_s[2]))))
        res = {"views": nv, "grad_max_abs_over_max": worst, "stat_counters_equal": counters_equal, "stat_sums_close": sums_close,
               "visible_count": [int(got_n), int(want_n)], "allreduce_bytes": w.bucket.nbytes(),
               "ok": bool(worst < 2e-4 and got_n == want_n and counters_equal and sums_close),
               "what": "rank r renders view r of a " + str(nv) + "-view ring (NCCL: all_gather of rendered images for the cross-view term, in-place "
                       "gradient all-reduce, last-view statistics broadcast, int64 count all-reduce) vs rank 0 rendering every view alone"}
    pc.feat_planes.Q0 = q0
    dist.barrier()
    return res


def run_ours(args):
    import torch.distributed as dist
    from splatco_b200 import _lib, decode, profiling

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    L = _lib.lib()
    w = Workload(args, args.workload, device, rank, world)
    w.keep_outputs = bool(args.dump_outputs) and rank == 0
    cfg, mv = w.cfg, w.mv
    H, W = cfg["H"], cfg["W"]
    # the GPU side of the `parity` block: view 0 at Q0 = 0 BEFORE anything updates the parameters (compared with the
    # oracle's rendering of the same view in the cpu_baseline leg)
    parity_gpu = None
    if world == 1 and not args.no_cpu:
        parity_gpu = parity_render(w)

    warm = max(args.warmup, 3)
    # the clock sampler starts BEFORE the warm-up: nvidia-smi's start-up (NVML initialisation) stalls the GPU for tens
    # of ms on some boxes, which otherwise lands inside the first timed loop; it keeps sampling through the timed region
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.5)
    for _ in range(warm):
        w.step(False)
    # ... and on until torch's caching allocator is in steady state: a cudaMalloc inside the timed region costs 10-100 ms when
    # peer access is enabled (multi-GPU), and the pool keeps growing by a block every few steps for a while (how many
    # buffers of a size are alive at once depends on how far the host runs ahead)
    warm_extra = warm_until_quiescent(w, device, world)
    # the training-time plane-feature noise of a decode call is seeded from torch's seed and a per-process call counter:
    # fixing both here makes the timed steps' inputs depend on the arguments only, not on the process or on how many
    # warm-up steps the allocator needed
    torch.manual_seed(0)
    decode._noise_calls = 0
    launches0 = L.splatco_launch_count()
    ms_dev = w.timed(w.step, args.steps, False)
    launches = L.splatco_launch_count() - launches0
    dumped = w.outputs() if w.keep_outputs else None
    w.keep_outputs, w.last = False, None
    ms_e2e = w.timed(w.step, args.steps, True)
    clocks = sampler.stop() if rank == 0 else None
    # per-stage CUDA-event times come from a separate pass (two event records per stage would otherwise
    # sit inside the headline number); shares are relative to this pass's own step time.  The tensor-core MLP kernels
    # of the decode are bracketed by events inside the library in the same pass.
    L.splatco_decode_profile(1)
    with profiling.collect() as prof:
        ms_stage = w.timed(w.step, args.steps, False, tag="stage_pass")
    stage_sum = prof.summary()
    mlp_ms = None
    if L.splatco_decode_get_impl() == 2:
        import ctypes as C
        f_ms, b_ms = C.c_float(0), C.c_float(0)
        if L.splatco_decode_profile_read(C.byref(f_ms), C.byref(b_ms)) == 0:
            mlp_ms = (float(f_ms.value), float(b_ms.value))
    L.splatco_decode_profile(0)
    # whole training iteration (BASELINE metric "train it/s"): the same step + the optimizer update the reference performs
    # at train.py:310-312 (Adam over every parameter group, eps 1e-15, scene/gaussian_model.py:519-572), fused
    from splatco_b200.optim import FusedAdam
    opt = FusedAdam([{"params": [p], "lr": 1e-6, "name": f"p{i}"} for i, p in enumerate(w.params) if p.requires_grad], lr=0.0, eps=1e-15)

    def train_iter(host_inputs):
        loss = w.step(host_inputs)
        opt.step()
        return loss
    for _ in range(2):
        train_iter(False)
    launches_t0 = L.splatco_launch_count()
    ms_train = w.timed(train_iter, args.steps, True)
    launches_train = L.splatco_launch_count() - launches_t0
    del opt

    views = mv * world
    ms_step = ms_dev / args.steps
    check = multi_gpu_check(w) if world > 1 else None
    out = None
    if rank == 0:
        R, visited, live = w.instance_counts()
        M, V, N = w.info["M"], w.info["V"], cfg["N"]
        stages, alg_bytes, dom = stage_table(w, stage_sum, ms_stage, R, M, V)
        peak, peak_src = peaks()
        roof = None
        ncu = ncu_evidence()
        if dom:
            a = stages[dom]["alg_gbs"]
            ev = ncu.get(dom + "_kernel")
            roof = {"kernel": dom, "bound": "hbm", "achieved": a, "peak": peak, "unit": "GB/s",
                    "frac": round(a / peak, 4), "peak_source": peak_src,
                    "traffic": int(ev["dram_bytes"]) if ev else None,      # dram read+write per launch, ncu --set full
                    "traffic_source": ncu.get("_file") if ev else None,
                    "alg_bytes_per_launch": int(alg_bytes[dom])}
        # the blend is instruction-issue bound, not HBM bound (SURVEY §8d; ncu: DRAM < 2 % of peak): its honest roofline is
        # issue slots.  Work units: LIVE (pixel, instance) pairs (alpha >= 1/255 before the pixel terminates -- the pairs that
        # contribute and receive gradients); visited pairs = everything a per-pixel walk touches; slots = 256 R.
        blend = {"instances_R": int(R), "slots_256R": int(256 * R), "visited_pairs": int(visited), "live_pairs": int(live),
                 "live_frac_of_slots": round(live / max(256.0 * R, 1.0), 4)}
        sm_clock = (clocks or {}).get("sm_mhz") or 1965.0
        issue_peak = 148 * 4 * sm_clock * 1e6                          # warp instructions / s: 4 schedulers per SM, 1 per clock
        for k in ("blend_fwd", "blend_bwd"):
            if k in stages and live > 0:
                t = stages[k]["avg_ms"] * 1e-3
                e = {"ms": stages[k]["avg_ms"], "live_pairs_per_s": round(live / t, 1), "ns_per_live_pair_per_sm": round(t * 148 / live * 1e9, 4),
                     "issue_slots_per_live_pair": round(issue_peak * t / live, 3)}
                ev = ncu.get(k + "_kernel")
                if ev and ev.get("warp_instructions"):
                    e.update({"warp_instructions": int(ev["warp_instructions"]), "warp_instructions_per_live_pair": round(ev["warp_instructions"] / live, 3),
                              "lane_efficiency": round(ev.get("threads_per_instruction", 0.0) / 32.0, 3), "issue_active_pct": ev.get("issue_active_pct"),
                              "source": ncu.get("_file")})
                blend[k] = e
        if roof is not None and dom.startswith("blend"):
            roof["pairs_per_s"] = round(R * 256 / (stages[dom]["avg_ms"] * 1e-3), 1)
            roof["issue_slot_roofline"] = blend
        # the decode MLP runs on tcgen05 (3xTF32): algorithmic FLOPs counted once, against half the measured bf16 peak;
        # kernel time from THIS run's CUDA events (splatco_decode_profile)
        mlp = None
        if mlp_ms is not None and mlp_ms[0] > 0:
            pk, pk_src = _tf32_peak()
            flops = V * (32.5e3 + 5.5e3 * LEVEL)
            ach_f, ach_b = flops / (mlp_ms[0] * 1e-3) / 1e12, 2.0 * flops / (mlp_ms[1] * 1e-3) / 1e12 if mlp_ms[1] > 0 else None
            ev = ncu.get("dec2_mlp_fwd_kernel")
            mlp = {"kernel": "dec2_mlp_fwd_kernel", "bound": "tensor", "achieved": round(ach_f, 2), "peak": round(pk, 1), "unit": "TFLOP/s",
                   "frac": round(ach_f / pk, 4), "peak_source": pk_src, "kernel_ms": round(mlp_ms[0], 4), "time_source": "CUDA events around the kernel, this run",
                   "backward": {"kernel": "dec2_mlp_bwd_kernel", "kernel_ms": round(mlp_ms[1], 4), "achieved": round(ach_b, 2) if ach_b else None,
                                "frac": round(ach_b / pk, 4) if ach_b else None},
                   "tensor_pipe_active_pct": ev["tensor_active_pct"] if ev else None, "ncu_source": ncu.get("_file") if ev else None}
        out = {
            "metric": "fwd_bwd_ms_per_view", "value": round(ms_step / views, 4), "unit": "ms/view", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "warmup_extra": warm_extra, "ms_per_step": round(ms_step, 4), "higher_is_better": False,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["desc"], "path": "prefilter_voxel + render() drop-in: decode, preprocess, binning, blend, fwd+bwd",
                       "anchors": N, "visible_anchors": int(V), "gaussians": int(M), "instances_R": int(R),
                       "activate_level": LEVEL, "plane_size": cfg["plane_size"], "num_channels": cfg["C"], "Q0": 0.03,
                       "decode_impl": int(L.splatco_decode_get_impl()),
                       "mv": mv, "views_per_step": views, "loss": "0.8*L1 + 0.2*(1-SSIM) (fused kernels) + 0.01*mean(prod(scaling)) (" + ("torch ops" if args.torch_scaling_reg else "splatco scaling_reg kernel, no host sync in its backward") + "), train.py:192-196",
                       "l2": "per-step working set (planes + workspaces) exceeds the 126 MB L2; no explicit flush",
                       "parallelism": f"view-sharded dp{world}, NCCL grad all-reduce" if world > 1 else "single GPU"},
            "it_per_s": round(1000.0 / ms_step, 3),
            "e2e": {"value": round((ms_e2e / args.steps) / views, 4), "unit": "ms/view",
                    "h2d_bytes_per_step": int(mv * 3 * H * W * 4), "d2h_bytes_per_step": 4 + 8 * mv},
            "gpu_launches": int(launches),
            "train": {"it_per_s": round(1000.0 * args.steps / ms_train, 3), "ms_per_iter": round(ms_train / args.steps, 4),
                      "gpu_launches": int(launches_train),
                      "includes": "the e2e step (H2D ground truth, mv views fwd+bwd, loss read-back" + (", NCCL grad all-reduce" if world > 1 else "") +
                                  ") + FusedAdam update of every parameter (train.py:310-312), lr 1e-6"},
            "roofline": roof, "decode_mlp": mlp, "stages": stages, "clocks": clocks,
            "per_step_ms": w.host_ms,
        }
        if w.bucket is not None:
            out["config"]["allreduce_bytes_per_step"] = w.bucket.nbytes()
        if check is not None:
            out["multi_gpu_check"] = check
        if world == 1 and not args.no_gpu_baseline:
            out["gpu_baseline"] = gpu_baseline(w)
    # ---- other BASELINE configs in the same line: C3 on one GPU, C4 (one view per GPU = its mv = 8 batch) on eight ----
    subs = {}
    del w
    gc.collect()
    torch.cuda.empty_cache()
    if args.workload == "c2" and not args.no_sub:
        if world == 1:
            subs["c3"] = sub_record(args, "c3", device, rank, world)
        elif world == 8:
            subs["c4"] = sub_record(args, "c4", device, rank, world)
    if rank == 0:
        if subs:
            out["sub_records"] = subs
        if world == 1 and not args.no_cpu:
            base, parity = cpu_baseline(cfg, parity_gpu)
            out["cpu_baseline"] = base
            out["parity"] = parity
        if dumped is not None:
            dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def parity_render(w: Workload):
    """View 0 of the workload at Q0 = 0 through the product path; host copies of what the oracle leg compares."""
    from splatco_b200.gaussian_renderer import prefilter_voxel, render
    pc = w.pc
    q0 = pc.feat_planes.Q0
    pc.feat_planes.Q0 = 0.0
    with torch.no_grad():
        vm = prefilter_voxel(w.cams[0], pc, PIPE, w.bg)
        pkg = render(w.cams[0], pc, PIPE, w.bg, visible_mask=vm)
        res = {"vm": vm.cpu().numpy(), "image": pkg["render"].cpu().numpy(), "radii": pkg["radii"].cpu().numpy(),
               "mask": pkg["selection_mask"].cpu().numpy()}
    pc.feat_planes.Q0 = q0
    return res


# ---- CPU oracle port (cpu_baseline leg and --impl reference) -------------------------------------------
class _CpuScene:
    def __init__(self, cfg):
        self.cfg = cfg
        self.pc = build_model(cfg, "cpu")
        self.pc.feat_planes.Q0 = 0.0
        self.cams, self.gts = build_views(cfg)
        self.p = {"feat." + k: v for k, v in self.pc.feat_planes._feat.state_dict().items()}
        for name in ("mlp_opacity", "mlp_cov", "mlp_color"):
            self.p.update({f"{name}.{k}": v for k, v in getattr(self.pc, name).state_dict().items()})
        for k, v in self.p.items():
            if v.dtype.is_floating_point and "running" not in k and "xyz_m" not in k:
                v.requires_grad_(True)

    def view(self, i):
        """prefilter + decode + rasterize forward, L1 gradient, rasterize + decode backward; returns seconds."""
        from oracle import decode_oracle as D
        from oracle import raster as R
        cfg, pc = self.cfg, self.pc
        cam, gt = self.cams[i % len(self.cams)], self.gts[i % len(self.gts)].numpy()
        H, W = cfg["H"], cfg["W"]
        tx, ty = math.tan(cam.FoVx * 0.5), math.tan(cam.FoVy * 0.5)
        view, proj = cam.world_view_transform.numpy(), cam.full_proj_transform.numpy()
        bg = np.ones(3, np.float32)
        t0 = time.perf_counter()
        scaling = torch.exp(pc._scaling)
        radii = R.visible_filter(pc._anchor.detach().numpy(), scaling.detach().numpy()[:, :3],
                                 torch.nn.functional.normalize(pc._rotation).numpy(), 1.0, view, proj, tx, ty, H, W)
        vis = torch.from_numpy(radii > 0)
        xyz, color, opacity, scl, rot, nopac, mask = D.decode(self.p, pc._anchor_feat, pc._anchor, pc._offset, scaling, vis,
                                                              cam.camera_center, LEVEL, cfg["K"])
        a = [t.detach().numpy() for t in (xyz, color, opacity, scl, rot)]
        fw = R.rasterize_forward(a[0], a[1], a[2], a[3], a[4], 1.0, view, proj, tx, ty, H, W, bg)
        dL = (np.sign(fw["image"] - gt) / (3.0 * H * W)).astype(np.float32)
        g = R.rasterize_backward(fw, a[0], a[1], a[3], a[4], 1.0, view, proj, tx, ty, H, W, bg, dL)
        outs = [xyz, color, opacity, scl, rot]
        grads = [torch.from_numpy(g[k]) for k in ("means3D", "colors", "opacities", "scales", "rotations")]
        torch.autograd.backward(outs, grads)
        for t in [pc._anchor_feat, pc._anchor, pc._offset, pc._scaling] + list(self.p.values()):
            t.grad = None
        self.last = {"vis": vis.numpy(), "fw": fw, "mask": mask.numpy(), "nopac": nopac.detach().numpy()}
        return time.perf_counter() - t0


def parity_block(gpu, cpu, H, W):
    """The driver-run number checked against the oracle in the same run: forward of view 0 at Q0 = 0 (the test suite
    holds the backward: tests/test_parity_timed_gpu.py)."""
    fw = cpu["fw"]
    want_mask, got_mask = cpu["mask"], gpu["mask"]
    out = {"view": 0, "prefilter_mask_equal": bool(np.array_equal(gpu["vm"], cpu["vis"]))}
    if got_mask.shape != want_mask.shape:
        out["error"] = "visible-anchor counts differ"
        return out
    mism = got_mask != want_mask
    decided = np.abs(cpu["nopac"][:, 0]) > 1e-5
    out["mask_mismatch"] = int(mism.sum())
    out["mask_mismatch_decided"] = int((mism & decided).sum())
    full_g = np.zeros(got_mask.shape[0], np.int64); full_g[got_mask] = gpu["radii"]
    full_w = np.zeros(want_mask.shape[0], np.int64); full_w[want_mask] = fw["pr"].radii
    both = got_mask & want_mask
    rd = full_g[both] != full_w[both]
    out["gaussians"] = int(want_mask.sum())
    out["radii_equal"] = bool(not rd.any() and not mism.any())
    out["radii_mismatch"] = int(rd.sum())       # decode outputs of the two sides differ by fp32 rounding: see tests/test_parity_timed_gpu.py
    err = np.abs(gpu["image"] - fw["image"]).max(axis=0)
    fragile = fw["fragile"].copy()
    out["fragile_frac"] = round(float(fragile.mean()), 5)
    if rd.any():
        idx = np.nonzero(want_mask)[0]
        rows = np.searchsorted(idx, np.nonzero(both)[0][np.nonzero(rd)[0]])
        yy, xx = np.mgrid[0:H, 0:W]
        for r_ in rows[:64]:
            cx, cy = fw["pr"].xy[r_]
            rad = fw["pr"].radii[r_] + 17
            fragile |= (np.abs(xx - cx) <= rad) & (np.abs(yy - cy) <= rad)
    out["excluded_frac"] = round(float(fragile.mean()), 5)
    out["image_max_abs"] = float(err[~fragile].max())
    out["image_max_abs_excluded"] = float(err[fragile].max()) if fragile.any() else 0.0
    out["ok"] = bool(out["prefilter_mask_equal"] and out["mask_mismatch_decided"] == 0 and out["image_max_abs"] <= 1e-4
                     and out["image_max_abs_excluded"] <= 1e-2 and out["radii_mismatch"] <= max(2, int(2e-5 * out["gaussians"])))
    out["bars"] = "prefilter mask equal; opacity mask equal where |neural_opacity| > 1e-5; image <= 1e-4 off excluded pixels (oracle-fragile pairs, tiles of Gaussians whose radius differs by one), <= 1e-2 on them"
    return out


def cpu_baseline(cfg, parity_gpu=None):
    from oracle import raster as R
    torch.set_num_threads(os.cpu_count() or 1)
    sc = _CpuScene(cfg)
    dt = sc.view(0)
    base = {"value": round(dt * 1e3, 2), "unit": "ms/view", "cores": int(R.lib().oracle_get_threads()),
            "kind": "port", "sample": "1 view of the same workload, fwd+bwd: oracle/decode_oracle.py (torch CPU, "
                                      "autograd) + oracle/raster_oracle.c on all host threads"}
    parity = None
    if parity_gpu is not None:
        try:
            parity = parity_block(parity_gpu, sc.last, cfg["H"], cfg["W"])
        except Exception as e:
            parity = {"error": repr(e)[:200]}
    return base, parity


def run_reference(args):
    """Reference arm = the oracle port of the path on the host cores (see module doc)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import raster as R
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = WORKLOADS[args.workload]
    sc = _CpuScene(cfg)
    budget_s, t_start = 240.0, time.perf_counter()
    nwarm = min(args.warmup, 1)
    for i in range(nwarm):
        sc.view(i)
    times = []
    for i in range(args.steps):
        times.append(sc.view(i))
        if time.perf_counter() - t_start > budget_s:
            break
    ms = float(np.mean(times)) * 1e3
    cores = int(R.lib().oracle_get_threads())
    out = {"impl": "reference", "metric": "fwd_bwd_ms_per_view", "value": round(ms, 2), "unit": "ms/view",
           "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": len(times), "warmup": nwarm,
           "ms_per_step": round(ms, 2), "higher_is_better": False, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": {"workload": cfg["desc"], "path": "oracle port: prefilter + decode + rasterize, fwd+bwd, one view per step",
                      "anchors": cfg["N"], "mv": cfg["mv"], "activate_level": LEVEL},
           "cpu_baseline": {"value": round(ms, 2), "unit": "ms/view", "cores": cores, "kind": "port",
                            "sample": "one view of the workload per step (the reference's CUDA rasterizer is absent and "
                                      "has no CPU path; its Python decode cannot travel): oracle port on all host threads"},
           "e2e": {"value": round(ms, 2), "unit": "ms/view", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (and the parity block computed with it)")
    ap.add_argument("--no-sub", action="store_true", help="skip the sub-records of the other BASELINE configs (c3 at 1 GPU, c4 at 8)")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="skip the same-GPU comparators")
    ap.add_argument("--level", type=int, default=2, choices=[0, 1, 2],
                    help="activate_level of the feature planes: 2 = steady state after iteration 21 000 (default, the headline), "
                         "0 = the first 12 000 iterations (train.py:305-307, SURVEY §8d times both)")
    ap.add_argument("--torch-scaling-reg", action="store_true",
                    help="scaling regulariser with torch ops as train.py:195 writes it (its prod backward syncs with the host every view)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's images, loss and parameter gradients to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed (--impl ours)")
    global LEVEL
    LEVEL = args.level
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
