#!/usr/bin/env python
"""Cost of the image-weight gradient (RasterConfig.differentiable_weight) in the backward rasterizer.  For each feature
width F, the same projected scene and tile lists are rasterized forward and backward in three ways:

  plain    flag off, loss sum(image G)                       gs_raster_bwd, F channels
  weight   flag on, loss sum(image G) + sum(W Gw)            gs_raster_bwd_with_weight, F channels
  ones     flag off, features [f, 1], loss sum(image [G, Gw]) gs_raster_bwd, F + 1 channels (the workaround)

Reported per arm: the device time of the backward entry point (CUDA events around the call: the backward kernels
plus, for F <= 7 without antialiasing, the moment pass), median over --iters interleaved repetitions.  The weight and ones arms must give the same gradients (checked, relative L2 printed).

  python benchmarks/weight_gradient.py [--iters 20] [--widths 3:bench,7:bench,34:c4,64:c4,256:c4]

F = 7 and F = 64 are where the workaround changes kernel family (narrow -> wide, wide -> extra-wide).  The card's name
and power limit are read in the same run and printed first.  Every scene's working set (2-3 M gaussians, 2K / 4K
images) exceeds the 126 MB L2.
"""
import argparse
import json
import statistics
import subprocess
import sys
from dataclasses import replace
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from taichi_gaussian_rasterizer_b200 import (RasterConfig, _native, map_to_tiles, rasterize_with_tiles,  # noqa: E402
                                             render_gaussians)
from taichi_gaussian_rasterizer_b200.synthetic import baseline_scene  # noqa: E402
from taichi_gaussian_rasterizer_b200.torch_lib.projection import ndc_depth  # noqa: E402

BWD = ("gs_raster_bwd", "gs_raster_bwd_with_weight")


def card():
  q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
  return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def rel_l2(a, b):
  return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--iters", type=int, default=20)
  ap.add_argument("--widths", default="3:bench,7:bench,34:c4,64:c4,256:c4", help="F:scene pairs")
  ap.add_argument("--stats", action="store_true", help="visibility and split / prune heuristics on")
  args = ap.parse_args()
  if not torch.cuda.is_available():
    raise SystemExit("weight_gradient.py measures on a CUDA device; none found")
  dev = torch.device("cuda:0")
  print(json.dumps(card()), flush=True)
  cfg = RasterConfig(compute_visibility=args.stats, compute_point_heuristic=args.stats)

  for item in args.widths.split(","):
    F, scene = int(item.split(":")[0]), item.split(":")[1]
    g, cam, spec = baseline_scene(scene)
    torch.manual_seed(1)
    g.feature = torch.rand(g.feature.shape[0], F)
    g, cam = g.to(device=dev), cam.to(device=dev)
    W, H = cam.image_size
    with torch.no_grad():
      out = render_gaussians(g, cam, cfg, use_sh=False)
      g2d = out.gaussians2d.contiguous()
      o2p, ranges = map_to_tiles(g2d, ndc_depth(out.point_depth, cam.near_plane, cam.far_plane), cam.image_size, cfg)
      ranges = ranges.view(-1, 2)
      feat = g.feature[out.points_in_view].contiguous()
    del out
    ones = torch.cat([feat, torch.ones_like(feat[:, :1])], dim=1)
    gi = torch.rand(H, W, F, device=dev) - 0.3
    gw = torch.rand(H, W, device=dev) - 0.3
    gi1 = torch.cat([gi, gw[..., None]], dim=-1)

    def step(arm):
      gd, fd = g2d.clone().requires_grad_(True), (ones if arm == "ones" else feat).clone().requires_grad_(True)
      c = replace(cfg, differentiable_weight=arm == "weight")
      r = rasterize_with_tiles(gd, fd, o2p, ranges, cam.image_size, c)
      if arm == "ones":
        loss = (r.image * gi1).sum()
      elif arm == "weight":
        loss = (r.image * gi).sum() + (r.image_weight * gw).sum()
      else:
        loss = (r.image * gi).sum()
      loss.backward()
      return gd.grad, fd.grad, r.point_heuristic

    with_ones = F + 1 <= 256   # the rasterizer's channel limit: at F = 256 the workaround does not exist
    arms = ["plain", "weight"] + (["ones"] if with_ones else [])
    row = {"F": F, "scene": scene, "image": [W, H], "visible": int(g2d.shape[0]), "overlaps": int(o2p.shape[0]),
           "stats": args.stats}
    if with_ones:
      gw_ = step("weight")
      go = step("ones")
      row["weight_vs_ones_rel_l2"] = {"gaussians": rel_l2(gw_[0], go[0]), "features": rel_l2(gw_[1], go[1][:, :F])}
      if args.stats:
        row["weight_vs_ones_rel_l2"]["heuristic"] = rel_l2(gw_[2], go[2])
      del gw_, go
    for arm in arms:   # warm-up: module loading, allocator pools
      step(arm)
    torch.cuda.synchronize()
    times = {arm: [] for arm in arms}
    for _ in range(args.iters):
      for arm in arms:   # interleaved, so that drift of the shared machine hits every arm alike
        timer = _native.set_stage_timer(_native.StageTimer())
        step(arm)
        s = timer.summary()
        _native.set_stage_timer(None)
        times[arm].append(sum(s[k][1] for k in BWD if k in s))
    for arm in arms:
      row[arm + "_bwd_ms"] = round(statistics.median(times[arm]), 3)
      row[arm + "_bwd_ms_min"] = round(min(times[arm]), 3)
    row["weight_over_plain"] = round(row["weight_bwd_ms"] / row["plain_bwd_ms"], 3)
    if with_ones:
      row["ones_over_plain"] = round(row["ones_bwd_ms"] / row["plain_bwd_ms"], 3)
    print(json.dumps(row), flush=True)
    del g, gi, gw, gi1, feat, ones, g2d
    torch.cuda.empty_cache()


if __name__ == "__main__":
  main()
