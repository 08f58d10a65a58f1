"""RasterConfig.differentiable_weight: image_weight W = sum_i w_i as a differentiable output, in every backward kernel
family.  W is the blend of a constant feature 1, so the exact reference is the oracle rasterizing [features, 1] with the
image gradient [G, Gw]: its gaussian gradient and heuristics, its first F feature-gradient columns, and its channel F
(which equals image_weight)."""
from dataclasses import replace

import pytest
import torch

import oracle
from oracle import torch_ref
from taichi_gaussian_rasterizer_b200 import CapturedStep, RasterConfig, rasterize_with_tiles, render_gaussians
from taichi_gaussian_rasterizer_b200.renderer import compute_depth_variance
from test_gpu_rasterizer import compare_forward_backward
from util import GRAD_REL_L2, IMAGE_REL_L2, rel_l2, scene2d, scene3d

pytestmark = pytest.mark.gpu


def compare_weight_gradient(cuda_device, seed, n, size, cfg, channels=3, scale=1.0, dtype=torch.float32):
  """loss = sum(image GI) + sum(W GW) on the GPU with differentiable_weight, against the oracle with a ones channel"""
  cfg = replace(cfg, differentiable_weight=True)
  F = channels
  g, depth, feat = scene2d(seed, n, size, channels=F, scale_factor=scale, dtype=dtype)
  o2p, ranges = oracle.map_to_tiles(g.float(), depth, size, cfg)
  torch.manual_seed(seed + 1)
  gi = torch.rand(size[1], size[0], F, dtype=dtype) - 0.3
  gw = torch.rand(size[1], size[0], dtype=dtype) - 0.3

  gr = g.clone().requires_grad_(True)
  fr = feat.clone().requires_grad_(True)
  ref = oracle.rasterize_with_tiles(gr, torch.cat([fr, torch.ones_like(fr[:, :1])], dim=1), o2p, ranges.view(-1, 2),
                                    size, cfg)
  (ref.image * torch.cat([gi, gw[..., None]], dim=-1)).sum().backward()

  gd, fd = g.to(cuda_device).requires_grad_(True), feat.to(cuda_device).requires_grad_(True)
  out = rasterize_with_tiles(gd, fd, o2p.to(cuda_device), ranges.view(-1, 2).to(cuda_device), size, cfg)
  assert out.image_weight.requires_grad
  ((out.image * gi.to(cuda_device)).sum() + (out.image_weight * gw.to(cuda_device)).sum()).backward()

  errs = dict(image=rel_l2(out.image, ref.image[..., :F]), weight=rel_l2(out.image_weight, ref.image[..., F]),
              gaussians=rel_l2(gd.grad, gr.grad), features=rel_l2(fd.grad, fr.grad))
  if cfg.compute_point_heuristic:
    errs["heuristic"] = rel_l2(out.point_heuristic, ref.point_heuristic)
  print(errs)
  assert errs["image"] < IMAGE_REL_L2 and errs["weight"] < IMAGE_REL_L2, errs
  assert errs["gaussians"] < GRAD_REL_L2 and errs["features"] < GRAD_REL_L2, errs
  if cfg.compute_point_heuristic:
    assert errs["heuristic"] < 10 * GRAD_REL_L2, errs
  if cfg.compute_visibility:
    assert rel_l2(out.visibility, ref.visibility) < GRAD_REL_L2
  return errs


@pytest.mark.parametrize("channels", [1, 3, 5, 7])
@pytest.mark.parametrize("stats", [False, True])
def test_narrow(cuda_device, channels, stats):
  cfg = RasterConfig(compute_visibility=stats, compute_point_heuristic=stats)
  compare_weight_gradient(cuda_device, 10 + channels, 3000, (200, 150), cfg, channels=channels, scale=2.0)


@pytest.mark.parametrize("channels", [3, 5])
def test_narrow_antialiased(cuda_device, channels):
  cfg = RasterConfig(antialias=True, compute_visibility=True, compute_point_heuristic=True)
  compare_weight_gradient(cuda_device, 20 + channels, 3000, (200, 150), cfg, channels=channels, scale=2.0)


@pytest.mark.parametrize("channels", [8, 12, 34, 64])
def test_wide(cuda_device, channels):
  cfg = RasterConfig(compute_visibility=True, compute_point_heuristic=True)
  compare_weight_gradient(cuda_device, 30 + channels, 1500, (160, 112), cfg, channels=channels, scale=2.0)


@pytest.mark.parametrize("channels", [65, 128, 256])
def test_xwide(cuda_device, channels):
  cfg = RasterConfig(compute_visibility=True, compute_point_heuristic=True)
  compare_weight_gradient(cuda_device, 40 + channels, 1500, (160, 112), cfg, channels=channels, scale=2.0)


@pytest.mark.parametrize("channels", [3, 34])
def test_multi_batch_tile(cuda_device, channels):
  """tiles with several hundred to over a thousand overlaps: many staged batches, saturation exits"""
  cfg = RasterConfig(compute_visibility=True, compute_point_heuristic=True)
  compare_weight_gradient(cuda_device, 50 + channels, 4000, (64, 64), cfg, channels=channels, scale=6.0)


@pytest.mark.parametrize("tile,antialias,dtype", [(8, False, torch.float32), (32, False, torch.float32),
                                                  (8, True, torch.float32), (16, False, torch.float64),
                                                  (32, True, torch.float64)])
def test_generic(cuda_device, tile, antialias, dtype):
  cfg = RasterConfig(tile_size=tile, pixel_stride=(1, 1), antialias=antialias, compute_point_heuristic=True)
  compare_weight_gradient(cuda_device, 60 + tile, 2000, (150, 100), cfg, channels=3, scale=2.0, dtype=dtype)


@pytest.mark.parametrize("antialias", [False, True])
def test_gradcheck_image_and_weight(cuda_device, antialias):
  """float64 gradcheck of (image, image_weight) on one 8x8 tile, as test_rasterizer_gradcheck does for the image"""
  config = RasterConfig(tile_size=8, pixel_stride=(1, 1), antialias=antialias, differentiable_weight=True)
  torch.manual_seed(0)
  for seed in torch.randint(0, 1000, (10,)):
    torch.manual_seed(int(seed))
    n = int(torch.randint(1, 50, (1,)))
    channels = int(torch.randint(1, 4, (1,)))
    g, _, feat = scene2d(int(seed), n, (8, 8), channels=channels, alpha_range=(0.2, 0.8), dtype=torch.float64)
    g, feat = g.to(cuda_device), feat.to(cuda_device)
    o2p = torch.arange(0, n, device=cuda_device, dtype=torch.int32)
    ranges = torch.tensor([[0, n]], device=cuda_device, dtype=torch.int32)

    def render(mean, axis, sigma, alpha, colors):
      out = rasterize_with_tiles(torch.cat([mean, axis, sigma, alpha], dim=-1), colors, o2p, ranges, (8, 8), config)
      return out.image, out.image_weight

    inputs = (g[:, 0:2].requires_grad_(True), g[:, 2:4].requires_grad_(True), g[:, 4:6].requires_grad_(True),
              g[:, 6:7].requires_grad_(True), feat.requires_grad_(True))
    torch.autograd.gradcheck(render, inputs, eps=1e-6, check_grad_dtypes=True, check_undefined_grad=False,
                             nondet_tol=1e-9)


@pytest.mark.parametrize("channels", [3, 34, 128])
def test_flag_without_weight_in_loss(cuda_device, channels):
  """flag on, loss on the image only: the same image as flag off, gradients equal up to the order of atomic adds"""
  size = (160, 112)
  cfg = RasterConfig(compute_visibility=True, compute_point_heuristic=True)
  g, depth, feat = scene2d(80 + channels, 1500, size, channels=channels, scale_factor=2.0)
  o2p, ranges = oracle.map_to_tiles(g, depth, size, cfg)
  o2p, ranges = o2p.to(cuda_device), ranges.view(-1, 2).to(cuda_device)
  torch.manual_seed(1)
  gi = (torch.rand(size[1], size[0], channels) - 0.3).to(cuda_device)
  results = []
  for flag in (False, True):
    gd, fd = g.to(cuda_device).requires_grad_(True), feat.to(cuda_device).requires_grad_(True)
    out = rasterize_with_tiles(gd, fd, o2p, ranges, size, replace(cfg, differentiable_weight=flag))
    assert out.image_weight.requires_grad == flag
    (out.image * gi).sum().backward()
    results.append((out.image.detach(), out.image_weight.detach(), gd.grad, fd.grad, out.point_heuristic))
  off, on = results
  assert torch.equal(off[0], on[0]) and torch.equal(off[1], on[1])
  for a, b in zip(off[2:], on[2:]):
    assert rel_l2(b, a) < 2e-6


def test_flag_off_weight_not_differentiable(cuda_device):
  cfg = RasterConfig()
  out, _ = compare_forward_backward(cuda_device, 90, 500, (128, 96), cfg, check_grads=False)
  assert not out.image_weight.requires_grad
  quantile = RasterConfig(use_alpha_blending=False, differentiable_weight=True)
  g, depth, feat = scene2d(91, 500, (128, 96))
  o2p, ranges = oracle.map_to_tiles(g, depth, (128, 96), quantile)
  out = rasterize_with_tiles(g.to(cuda_device), feat.to(cuda_device).requires_grad_(True), o2p.to(cuda_device),
                             ranges.view(-1, 2).to(cuda_device), (128, 96), quantile)
  assert out.image.requires_grad and not out.image_weight.requires_grad   # W > 0 in quantile mode


def test_render_depth_and_composite_vs_oracle(cuda_device):
  """render_gaussians(render_depth=True): loss on the weight-normalised depth and on the image composited over a
  background, against the float64 pipeline with a ones channel in front of [depth, depth^2, features]"""
  cfg = RasterConfig(compute_visibility=True, compute_point_heuristic=True, differentiable_weight=True)
  size = (320, 240)
  g, cam = scene3d(3, 6000, image_size=size, scale_factor=0.5)
  gd, cd = g.to(device=cuda_device), cam.to(device=cuda_device)
  gd.requires_grad_(True)
  out = render_gaussians(gd, cd, cfg, use_sh=False, render_depth=True, render_median_depth=True)

  idx = out.points_in_view.cpu()
  ndc = torch_ref.ndc_depth(out.point_depth.detach().cpu(), cam.near_plane, cam.far_plane)
  o2p, ranges = oracle.map_to_tiles(out.gaussians2d.detach().cpu(), ndc, cam.image_size, cfg)
  gr = g.to(dtype=torch.float64).requires_grad_(True)
  cam64 = cam.to(dtype=torch.float64)
  pts_all, depth_all = torch_ref.project_all(*gr.shape_tensors(), cam64.T_camera_world, cam64.projection,
                                             cam.image_size, cfg.blur_cov, cfg.clamp_margin)
  pts, depth = pts_all[idx], depth_all[idx]
  feats = torch.cat([torch.ones_like(depth), depth, depth ** 2, gr.feature[idx]], dim=1)
  ref = oracle.rasterize_with_tiles(pts, feats, o2p, ranges.view(-1, 2), cam.image_size, cfg)
  ref_w = ref.image[..., 0]
  ref_depth, ref_var = compute_depth_variance(ref.image[..., 1:3], ref_w)
  ref_image = ref.image[..., 3:]

  torch.manual_seed(1)
  bg = torch.rand(3, dtype=torch.float64)
  gi = torch.rand(size[1], size[0], 3, dtype=torch.float64)
  gdep = torch.rand(size[1], size[0], dtype=torch.float64)
  composite = out.image + (1 - out.image_weight)[..., None] * bg.float().to(cuda_device)
  ((composite * gi.float().to(cuda_device)).sum() + (out.depth * gdep.float().to(cuda_device)).sum()).backward()
  ref_composite = ref_image + (1 - ref_w)[..., None] * bg
  ((ref_composite * gi).sum() + (ref_depth * gdep).sum()).backward()

  assert rel_l2(out.image_weight, ref_w) < 1e-4    # f32 path vs the float64 pipeline, as test_render_gaussians_vs_oracle
  assert rel_l2(out.depth, ref_depth) < 1e-4
  errs = {name: rel_l2(getattr(gd, name).grad, getattr(gr, name).grad)
          for name in ("position", "log_scaling", "rotation", "alpha_logit", "feature")}
  print(errs)
  # the bounds of test_render_gaussians_vs_oracle (position, scale and rotation go through the f32 projection)
  assert errs["feature"] < GRAD_REL_L2 and errs["alpha_logit"] < GRAD_REL_L2, errs
  assert errs["position"] < 5e-3 and errs["log_scaling"] < 0.3 and errs["rotation"] < 0.3, errs


def test_captured_step_random_background(cuda_device):
  """forward + backward through overlap_capacity= in a CapturedStep with a fresh random background per replay
  composited through image_weight: replay equals eager"""
  cfg = RasterConfig(compute_visibility=True, compute_point_heuristic=True, differentiable_weight=True)
  g, cam = scene3d(6, 4000, image_size=(160, 120), scale_factor=0.5)
  g, cam = g.to(device=cuda_device), cam.to(device=cuda_device)
  g.requires_grad_(True)
  names = ("position", "log_scaling", "rotation", "alpha_logit", "feature")
  params = [getattr(g, n) for n in names]
  torch.manual_seed(2)
  target = torch.rand(120, 160, 3, device=cuda_device)
  bg = torch.zeros(3, device=cuda_device)   # rewritten in place before every replay
  static_grads = [torch.zeros_like(p) for p in params]
  holder = {}

  def loss_of(out):
    composite = out.image + (1 - out.image_weight)[..., None] * bg
    return ((composite - target) ** 2).sum()

  def body():
    for p, b in zip(params, static_grads):
      b.zero_()
      p.grad = b
    out = render_gaussians(g, cam, cfg, use_sh=False, overlap_capacity=300_000)
    loss_of(out).backward()
    holder["image"], holder["weight"] = out.image, out.image_weight

  step = CapturedStep(body, device=cuda_device)
  for _ in range(2):
    bg.copy_(torch.rand(3, device=cuda_device))
    step.replay()
    torch.cuda.synchronize()
    got_image, got_weight = holder["image"].clone(), holder["weight"].clone()
    got = [b.clone() for b in static_grads]

    for p in params:
      p.grad = None
    out = render_gaussians(g, cam, cfg, use_sh=False)
    loss_of(out).backward()
    assert torch.equal(got_image, out.image) and torch.equal(got_weight, out.image_weight)
    for n, b, p in zip(names, got, params):
      assert rel_l2(b, p.grad) < 2e-6, (n, rel_l2(b, p.grad))
