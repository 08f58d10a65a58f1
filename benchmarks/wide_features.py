#!/usr/bin/env python
"""Wide feature images through render_gaussians on the config 4 scene (2 M gaussians, 3840x2160): F channels rendered
in one pass against the same frame done as 64-channel slices through the path that existed before 65..256 channels
were supported (one render_gaussians call per slice).  One JSON line per F:

  fwd_bwd_ms          forward + loss + backward of one frame, host clock around synchronised work (median of --iters)
  raster_fwd_ms /     device time of the gs_raster_fwd / gs_raster_bwd entry points (stage timer: pack, cull masks and
  raster_bwd_ms       the rasterizer kernel), summed over the slices for the sliced frame
  pairs_per_s         tile-list entries x 256 pixels / raster_fwd time: (pixel, gaussian) pairs the forward walks per
                      second, an upper bound on its blend evaluations
  sliced_*            the same for the 64-channel slices
  max_alloc_gb        torch.cuda.max_memory_allocated over one frame (feature tensor and scene included)

--dtypes float32,bfloat16 adds the feature dtype axis: the same frame with bfloat16 features (and so a bfloat16 image
and image gradient), the dtypes run alternately --rounds times and each key reported per dtype (median over rounds; no
sliced frames then).

  python benchmarks/wide_features.py [--features 64,128,256] [--iters 5] [--n 2000000] [--dtypes float32,bfloat16]

The card's name and power limit are read in the same run and printed first.  The working set (2 M x 256 features,
a 4K x 256 image and its gradient) is far beyond the 126 MB L2, so no pass is served from a warm cache.
"""
import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from taichi_gaussian_rasterizer_b200 import RasterConfig, _native, map_to_tiles, render_gaussians  # noqa: E402
from taichi_gaussian_rasterizer_b200.synthetic import baseline_scene  # noqa: E402
from taichi_gaussian_rasterizer_b200.torch_lib.projection import ndc_depth  # noqa: E402


def card():
  q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
  return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--features", default="64,128,256")
  ap.add_argument("--iters", type=int, default=5)
  ap.add_argument("--n", type=int, default=None, help="gaussians (default: the config 4 scene's 2 M)")
  ap.add_argument("--dtypes", default="float32", help="feature dtypes, e.g. float32,bfloat16")
  ap.add_argument("--rounds", type=int, default=3, help="alternations of the dtypes (with more than one)")
  args = ap.parse_args()
  dtypes = [getattr(torch, d) for d in args.dtypes.split(",")]
  if not torch.cuda.is_available():
    raise SystemExit("wide_features.py measures on a CUDA device; none found")
  dev = torch.device("cuda:0")
  print(json.dumps(card()), flush=True)
  cfg = RasterConfig()

  for F in [int(f) for f in args.features.split(",")]:
    g, cam, spec = baseline_scene("c4", n=args.n)
    torch.manual_seed(1)
    g.feature = torch.rand(g.feature.shape[0], F)
    g, cam = g.to(device=dev), cam.to(device=dev)
    g.requires_grad_(True)
    W, H = cam.image_size
    gi = torch.rand(H, W, F, device=dev) - 0.3
    if len(dtypes) > 1:
      print(json.dumps(dtype_rows(g, cam, cfg, gi, F, dtypes, args)), flush=True)
      del g, gi
      torch.cuda.empty_cache()
      continue

    def frame(sliced):
      for n in ("position", "log_scaling", "rotation", "alpha_logit", "feature"):
        getattr(g, n).grad = None
      if not sliced:
        out = render_gaussians(g, cam, cfg, use_sh=False)
        (out.image * gi).sum().backward()
        return out
      for c in range(0, F, 64):   # one call per slice: projection, tile map and both rasterizer passes each time
        part = g.replace(feature=g.feature[:, c:c + 64])
        out = render_gaussians(part, cam, cfg, use_sh=False)
        (out.image * gi[..., c:c + 64]).sum().backward()
      return out

    row = {"F": F, "image": [W, H], "n": g.position.shape[0]}
    for sliced in ((False, True) if F > 64 else (False,)):
      key = "sliced_" if sliced else ""
      for _ in range(2):
        out = frame(sliced)
      torch.cuda.synchronize()
      if not sliced:
        with torch.no_grad():
          K = map_to_tiles(out.gaussians2d, ndc_depth(out.point_depth, cam.near_plane, cam.far_plane), cam.image_size,
                           cfg)[0].shape[0]
        row["overlaps"] = int(K)
      times = []
      for _ in range(args.iters):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        frame(sliced)
        torch.cuda.synchronize()
        times.append((time.perf_counter() - t0) * 1e3)
      timer = _native.set_stage_timer(_native.StageTimer())
      for _ in range(args.iters):
        frame(sliced)
      summary = timer.summary()
      _native.set_stage_timer(None)
      fwd = summary["gs_raster_fwd"][1] / args.iters
      bwd = summary["gs_raster_bwd"][1] / args.iters
      row[key + "fwd_bwd_ms"] = round(statistics.median(times), 3)
      row[key + "fwd_bwd_ms_min"] = round(min(times), 3)
      row[key + "raster_fwd_ms"] = round(fwd, 3)
      row[key + "raster_bwd_ms"] = round(bwd, 3)
      row[key + "pairs_per_s"] = float(f"{row['overlaps'] * 256 * (F // 64 if sliced else 1) / (fwd * 1e-3):.4g}")
    print(json.dumps(row), flush=True)
    del g, gi
    torch.cuda.empty_cache()


def time_frame(g, cam, cfg, gi, iters):
  """one dtype's frame: host-clock ms of forward + loss + backward, stage-timer ms of the two rasterizer calls, peak
  allocation"""
  def frame():
    for n in ("position", "log_scaling", "rotation", "alpha_logit", "feature"):
      getattr(g, n).grad = None
    out = render_gaussians(g, cam, cfg, use_sh=False)
    (out.image * gi).sum().backward()

  frame()
  torch.cuda.synchronize()
  torch.cuda.reset_peak_memory_stats()
  frame()
  torch.cuda.synchronize()
  peak = torch.cuda.max_memory_allocated()
  times = []
  for _ in range(iters):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    frame()
    torch.cuda.synchronize()
    times.append((time.perf_counter() - t0) * 1e3)
  timer = _native.set_stage_timer(_native.StageTimer())
  for _ in range(iters):
    frame()
  summary = timer.summary()
  _native.set_stage_timer(None)
  return dict(fwd_bwd_ms=statistics.median(times), raster_fwd_ms=summary["gs_raster_fwd"][1] / iters,
              raster_bwd_ms=summary["gs_raster_bwd"][1] / iters, max_alloc_gb=peak / 1e9)


def dtype_rows(g, cam, cfg, gi, F, dtypes, args):
  """the frame with each feature dtype, the dtypes alternating round by round"""
  feature = g.feature.detach()
  views = {}
  for d in dtypes:   # one copy of the features (and of the image gradient) per dtype, made once
    gd = g.replace(feature=feature.to(d)).detach()
    gd.requires_grad_(True)
    views[d] = (gd, gi.to(d))
  del g
  runs = {d: [] for d in dtypes}
  for _ in range(args.rounds):
    for d in dtypes:
      runs[d].append(time_frame(views[d][0], cam, cfg, views[d][1], args.iters))
  row = {"F": F, "image": list(cam.image_size), "n": feature.shape[0]}
  for d in dtypes:
    name = str(d).replace("torch.", "")
    for k in runs[d][0]:
      row[f"{name}_{k}"] = round(statistics.median(r[k] for r in runs[d]), 3)
  return row


if __name__ == "__main__":
  main()
