"""The bench step at SH degree 0, 1, 2 and 3: ms per frame, and CUDA-event times of the SH kernels with their
algorithmic bytes and share of HBM peak.

  python benchmarks/sh_degrees.py [--degrees 0 1 2 3] [--steps 10] [--warmup 3] [--no-graph] [--root DIR] [--out FILE]

Scene: bench.py's (3 M gaussians, 2048x1365, tile 16, 8 views, two view streams); degree d keeps the first (d+1)^2
coefficients of its degree-3 features.  The step is bench.py's: inside GradientBucket.fused_accumulation(),
colours from evaluate_sh_views, L1 loss, backward, flush; "eager" through the default render_gaussians (host
read-backs), "graph" through render_gaussians(..., overlap_capacity=) captured in one CUDA graph (CapturedStep).
Where a tree cannot batch a degree (evaluate_sh_views refuses it) the step renders that degree with per-view colours
and says so; where it cannot capture it, the graph time is null.  ``--root`` imports the package from another
checkout (its own build), so two trees can be compared by alternating processes.

Bytes are the DESIGN.md §3 formulas with C = 3 and D = (d+1)^2: gs_sh_fwd_views N(4CD + 12 + 12 views) per batch,
gs_sh_bwd_stage 32V + 12N per view, gs_sh_bwd_flush N(12 views + 12 + 4CD) per batch (the first flush of a batch
overwrites), dense backward (coefficient gradient from the forward output, as render_gaussians takes it without a
bucket) 44V + 4CD N per view.  Share of peak: bytes / time against 6552 GB/s (the HBM peak DESIGN.md uses).
"""
import argparse
import ctypes
import json
import subprocess
import sys
import time
from pathlib import Path

import torch

HBM_PEAK = 6552e9


def card():
  name = torch.cuda.get_device_name(0)
  try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, text=True, timeout=20).stdout.strip()
  except Exception as e:   # noqa: BLE001
    q = f"nvidia-smi unavailable ({e})"
  return {"device": name, "nvidia_smi": q}


def event_ms(fn, reps):
  """Mean CUDA-event time of fn() over reps calls (after one warm-up call)."""
  fn()
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  a.record()
  for _ in range(reps):
    fn()
  b.record()
  torch.cuda.synchronize()
  return a.elapsed_time(b) / reps


def kernel_times(N, gaussians, cams, sh_params, reps):
  """CUDA-event times of the SH entry points on this degree's tensors, with bytes and share of peak; None where the
  library refuses the shape."""
  from taichi_gaussian_rasterizer_b200 import RasterConfig
  from taichi_gaussian_rasterizer_b200.perspective.projection import project_to_image
  dev = sh_params.device
  n, k, d = sh_params.shape
  views = len(cams)
  cd = k * d
  positions = gaussians.position.detach().contiguous()
  cam_pos = [c.camera_position.detach().contiguous() for c in cams]
  with torch.no_grad():
    _, _, idx = project_to_image(gaussians, cams[0], RasterConfig(tile_size=16))
  V = int(idx.shape[0])
  out = {"N": n, "V_view0": V, "D": d}

  def record(name, fn, nbytes, per):
    try:
      ms = event_ms(fn, reps)
    except RuntimeError as e:
      out[name] = {"ms": None, "error": str(e).splitlines()[0][:160]}
      return
    out[name] = {"ms": round(ms, 4), "per": per, "bytes": int(nbytes), "GB_per_s": round(nbytes / ms / 1e6, 1),
                 "fraction_of_6552": round(nbytes / ms / 1e6 / (HBM_PEAK / 1e9), 3)}

  outs = [torch.empty((n, k), device=dev) for _ in range(views)]
  arr = ctypes.c_void_p * views
  cam_arr = arr(*[c.data_ptr() for c in cam_pos])
  p_views = N.GsSHParams(N.GS_F32, k, d, 1, n, 0, 0, 0)
  record("gs_sh_fwd_views", lambda: N.call("gs_sh_fwd_views", ctypes.byref(p_views), ctypes.c_int32(views),
                                            N.ptr(sh_params), N.ptr(positions), cam_arr,
                                            arr(*[o.data_ptr() for o in outs]), N.stream_ptr(dev)),
         n * (4 * cd + 12 + 12 * views), f"batch of {views} views")

  fwd = outs[0][idx].contiguous()
  gout = torch.rand_like(fwd) - 0.3
  staged = [torch.empty((n, k), device=dev) for _ in range(views)]
  p_stage = N.GsSHParams(N.GS_F32, k, d, 1, n, V, 1, 1)

  def stage_batch():
    for s in staged:
      N.call("gs_sh_bwd_stage", ctypes.byref(p_stage), N.ptr(fwd), N.ptr(idx), N.ptr(gout), N.ptr(s), N.stream_ptr(dev))
  record("gs_sh_bwd_stage", stage_batch, views * (32 * V + 12 * n), f"batch of {views} views")

  # the sink as fused_accumulation() has it: the SH slice of the bench bucket, 11 N floats in
  flat = torch.empty(11 * n + n * cd, device=dev)
  sink = flat[11 * n:].view(n, k, d)
  p_flush = N.GsSHParams(N.GS_F32, k, d, 1, n, 0, 0, 1)
  record("gs_sh_bwd_flush", lambda: N.call("gs_sh_bwd_flush", ctypes.byref(p_flush), ctypes.c_int32(views),
                                            arr(*[s.data_ptr() for s in staged]), cam_arr, N.ptr(positions),
                                            N.ptr(sink), N.stream_ptr(dev)),
         n * (12 * views + 12 + 4 * cd), f"batch of {views} views (overwrite)")
  out["flush_sink_16B_aligned"] = sink.data_ptr() % 16 == 0

  g_params = torch.empty_like(sh_params)
  p_dense = N.GsSHParams(N.GS_F32, k, d, 1, n, V, 0, 1)
  record("gs_sh_bwd dense (from forward output)",
         lambda: N.call("gs_sh_bwd", ctypes.byref(p_dense), N.ptr(fwd), N.ptr(positions), N.ptr(idx),
                        N.ptr(cam_pos[0]), N.ptr(gout), N.ptr(g_params), N.ptr(None), N.ptr(None), N.stream_ptr(dev)),
         44 * V + 4 * cd * n, "view")
  return out


def run_degree(args, degree, gaussians_cpu, cameras):
  from taichi_gaussian_rasterizer_b200 import (CapturedStep, RasterConfig, evaluate_sh_views, overlap_capacity_for,
                                               render_gaussians)
  from taichi_gaussian_rasterizer_b200.distributed import GradientBucket, run_views
  dev = torch.device("cuda", 0)
  D = (degree + 1) ** 2
  g = gaussians_cpu.to(device=dev)
  g.feature = g.feature[:, :, :D].contiguous()
  g.requires_grad_(True)
  params = [g.position, g.log_scaling, g.rotation, g.alpha_logit, g.feature]
  bucket = GradientBucket(params)
  cfg = RasterConfig(tile_size=16)
  cams = [c.to(device=dev) for c in cameras]
  w, h = cams[0].image_size
  torch.manual_seed(1234)
  targets = [torch.rand(h, w, 3, device=dev) for _ in cams]
  streams = [torch.cuda.Stream(device=dev) for _ in range(2)]
  result = {"degree": degree, "D": D}
  try:
    evaluate_sh_views(g.feature, g.position, [cams[0].camera_position])
    batched = True
  except AssertionError:
    batched = False
  result["sh_colours"] = "evaluate_sh_views (batched)" if batched else "per view (evaluate_sh_views refuses this degree)"
  capacity = {"value": None}

  def step(static):
    with bucket.fused_accumulation():
      bucket.zero_()
      colors = (evaluate_sh_views(g.feature, g.position, [c.camera_position for c in cams]) if batched
                else [None] * len(cams))

      def view(i):
        kw = dict(overlap_capacity=capacity["value"]) if static else {}
        out = render_gaussians(g, cams[i], cfg, use_sh=True, sh_colors=colors[i], **kw)
        loss = torch.nn.functional.l1_loss(out.image, targets[i])
        loss.backward()
        return loss.detach()
      total = run_views(len(cams), view, streams)
      bucket.flush()
    return total

  def timed(fn):
    for _ in range(args.warmup):
      fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    a.record()
    for _ in range(args.steps):
      fn()
    b.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3 / args.steps
    return a.elapsed_time(b) / args.steps, wall

  ms, wall = timed(lambda: step(False))
  result["eager_ms_per_frame"] = round(ms / len(cams), 4)
  result["eager_wall_ms_per_frame"] = round(wall / len(cams), 4)
  result["graph_ms_per_frame"] = None
  if args.graph:
    try:
      capacity["value"] = overlap_capacity_for(g, cams, cfg)
      captured = CapturedStep(lambda: step(True), device=dev)
      ms, wall = timed(captured.replay)
      result["graph_ms_per_frame"] = round(ms / len(cams), 4)
      result["graph_wall_ms_per_frame"] = round(wall / len(cams), 4)
    except (AssertionError, RuntimeError) as e:
      result["graph_error"] = f"{type(e).__name__}: {str(e).splitlines()[0][:200] if str(e) else ''}"
  from taichi_gaussian_rasterizer_b200 import _native as N
  result["kernels"] = kernel_times(N, g, cams, g.feature.detach(), args.kernel_reps)
  del bucket, g, params
  torch.cuda.empty_cache()
  return result


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--degrees", type=int, nargs="+", default=[0, 1, 2, 3])
  ap.add_argument("--steps", type=int, default=10)
  ap.add_argument("--warmup", type=int, default=3)
  ap.add_argument("--views", type=int, default=8)
  ap.add_argument("--num-gaussians", type=int, default=0)
  ap.add_argument("--kernel-reps", type=int, default=20)
  ap.add_argument("--no-graph", dest="graph", action="store_false", help="eager step only")
  ap.add_argument("--root", default=str(Path(__file__).resolve().parents[1]),
                  help="checkout whose package (and build) is imported")
  ap.add_argument("--label", default="")
  ap.add_argument("--out", default=None, help="also write the JSON result here")
  args = ap.parse_args()
  assert torch.cuda.is_available(), "sh_degrees.py measures on a CUDA device"
  root = Path(args.root).resolve()
  sys.path.insert(0, str(root))
  sys.path.insert(1, str(Path(__file__).resolve().parents[1]))   # bench.py's scene builder
  import taichi_gaussian_rasterizer_b200 as pkg
  assert Path(pkg.__file__).resolve().parent.parent == root, f"imported {pkg.__file__}, not from {root}"
  from bench import build_scene
  gaussians, cameras, spec = build_scene("bench", 0, args.views, args.num_gaussians or None, None)
  res = {"label": args.label, "root": str(root), **card(), "scene": {"N": int(gaussians.position.shape[0]),
         "image_size": list(cameras[0].image_size), "views": args.views, "steps": args.steps, "warmup": args.warmup},
         "degrees": []}
  for d in args.degrees:
    res["degrees"].append(run_degree(args, d, gaussians, cameras))
    print(json.dumps(res["degrees"][-1]), flush=True)
  if args.out:
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1))
  print(json.dumps({k: v for k, v in res.items() if k != "degrees"}))


if __name__ == "__main__":
  main()
