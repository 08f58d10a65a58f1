#!/usr/bin/env python
"""Device time of gs_raster_fwd / gs_raster_bwd on one view of a BASELINE scene (min / median over interleaved rounds).
Alternative kernels are A/B-timed as two library builds, each loaded in its own process with _native.use_library
(as benchmarks/fast_math_cost.py does).

  python benchmarks/variants.py [--scene bench] [--stats] [--iters 20]
"""
import argparse
import json
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from taichi_gaussian_rasterizer_b200 import (RasterConfig, _native, evaluate_sh_at, map_to_tiles,  # noqa: E402
                                             rasterize_with_tiles)
from taichi_gaussian_rasterizer_b200.perspective.projection import project_to_image  # noqa: E402
from taichi_gaussian_rasterizer_b200.synthetic import baseline_scene  # noqa: E402
from taichi_gaussian_rasterizer_b200.torch_lib.projection import ndc_depth  # noqa: E402


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--scene", default="bench")
  ap.add_argument("--stats", action="store_true")
  ap.add_argument("--no-stats", action="store_true", help="visibility / heuristics off even if the scene asks for them")
  ap.add_argument("--iters", type=int, default=10)
  ap.add_argument("--rounds", type=int, default=7)
  args = ap.parse_args()
  dev = torch.device("cuda:0")
  g, cam, spec = baseline_scene(args.scene)
  stats = (args.stats or bool(spec.get("stats"))) and not args.no_stats
  cfg = RasterConfig(compute_visibility=stats, compute_point_heuristic=stats)
  g, cam = g.to(device=dev), cam.to(device=dev)
  with torch.no_grad():
    g2d, depth, idx = project_to_image(g, cam, cfg)
    if spec.get("sh_degree") is not None:
      feats = evaluate_sh_at(g.feature, g.position, idx, cam.camera_position)
    else:
      feats = g.feature[idx]
    if spec.get("render_depth"):
      feats = torch.cat([depth, depth ** 2, feats], dim=1)
    o2p, ranges = map_to_tiles(g2d, ndc_depth(depth, cam.near_plane, cam.far_plane), cam.image_size, cfg)
  feats = feats.contiguous()
  torch.manual_seed(0)
  gi = torch.rand(cam.image_size[1], cam.image_size[0], feats.shape[1], device=dev) - 0.3

  def step():
    a, b = g2d.detach().clone().requires_grad_(True), feats.detach().clone().requires_grad_(True)
    out = rasterize_with_tiles(a, b, o2p, ranges.view(-1, 2), cam.image_size, cfg)
    (out.image * gi).sum().backward()
    return out, a.grad, b.grad

  # boxes and clocks drift: the minimum / median over the rounds are reported
  for _ in range(3):
    step()
  times = {}
  for _ in range(args.rounds):
    step()
    torch.cuda.synchronize()
    timer = _native.set_stage_timer(_native.StageTimer())
    for _ in range(args.iters):
      step()
    for k, v in timer.summary().items():
      times.setdefault(k, []).append(v[1] / v[0])
    _native.set_stage_timer(None)
  ms = {k: {"min": round(min(v), 4), "median": round(sorted(v)[len(v) // 2], 4)} for k, v in times.items()}
  print(json.dumps({"scene": args.scene, "stats": stats, "K": int(o2p.shape[0]), "ms": ms}), flush=True)


if __name__ == "__main__":
  main()
