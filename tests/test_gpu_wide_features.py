"""Extra-wide feature images (65..256 channels) on the fast path, forward and backward in one pass: against the oracle,
against rendering 64-channel slices through the existing path (same image and gradients, different heuristics: the
heuristics are not linear in the channels), through render_gaussians eagerly and as a captured step, and the limits."""
import pytest
import torch

import oracle
from taichi_gaussian_rasterizer_b200 import CapturedStep, RasterConfig, rasterize_with_tiles, render_gaussians
from test_gpu_rasterizer import compare_forward_backward
from test_gpu_renderer import oracle_render
from util import GRAD_REL_L2, IMAGE_REL_L2, rel_l2, scene2d, scene3d

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("channels", [65, 96, 100, 128, 130, 256])
@pytest.mark.parametrize("stats", [False, True])
def test_xwide_vs_oracle(cuda_device, channels, stats):
  cfg = RasterConfig(compute_visibility=stats, compute_point_heuristic=stats)
  compare_forward_backward(cuda_device, 50 + channels, 1500, (160, 112), cfg, channels=channels, scale=2.0)


def test_xwide_multi_group_tile(cuda_device):
  """tiles with several hundred overlaps (many staged batches, saturation exits)"""
  cfg = RasterConfig(compute_visibility=True, compute_point_heuristic=True)
  out, _ = compare_forward_backward(cuda_device, 78, 3000, (64, 48), cfg, channels=130, scale=6.0)


def test_xwide_pixel_stride(cuda_device):
  cfg = RasterConfig(pixel_stride=(2, 2), compute_visibility=True, compute_point_heuristic=True)
  compare_forward_backward(cuda_device, 79, 1500, (160, 112), cfg, channels=200, scale=2.0)


def test_xwide_vs_slices(cuda_device):
  """256 channels in one pass equal four 64-channel passes in image and gradients; the heuristics differ from the
  sliced sum (aag^2 and |pgx| + |pgy| are not linear in the channels) and match the oracle."""
  F, size = 256, (160, 112)
  cfg = RasterConfig(compute_visibility=True, compute_point_heuristic=True)
  g, depth, feat = scene2d(91, 1500, size, channels=F, scale_factor=2.0)
  o2p, ranges = oracle.map_to_tiles(g, depth, size, cfg)
  o2p, ranges = o2p.to(cuda_device), ranges.view(-1, 2).to(cuda_device)
  torch.manual_seed(92)
  gi = (torch.rand(size[1], size[0], F) - 0.3).to(cuda_device)

  gd, fd = g.to(cuda_device).requires_grad_(True), feat.to(cuda_device).requires_grad_(True)
  full = rasterize_with_tiles(gd, fd, o2p, ranges, size, cfg)
  (full.image * gi).sum().backward()

  gs, fs = g.to(cuda_device).requires_grad_(True), feat.to(cuda_device).requires_grad_(True)
  images, heur = [], torch.zeros(g.shape[0], 2, device=cuda_device)
  for c in range(0, F, 64):
    part = rasterize_with_tiles(gs, fs[:, c:c + 64], o2p, ranges, size, cfg)
    (part.image * gi[..., c:c + 64]).sum().backward()
    images.append(part.image.detach())
    heur += part.point_heuristic
  assert rel_l2(full.image, torch.cat(images, dim=-1)) < IMAGE_REL_L2
  assert rel_l2(full.image_weight, part.image_weight) < IMAGE_REL_L2
  assert rel_l2(fd.grad, fs.grad) < GRAD_REL_L2
  assert rel_l2(gd.grad, gs.grad) < GRAD_REL_L2

  gr, fr = g.clone().requires_grad_(True), feat.clone().requires_grad_(True)
  ref = oracle.rasterize_with_tiles(gr, fr, o2p.cpu(), ranges.cpu(), size, cfg)
  (ref.image * gi.cpu()).sum().backward()
  assert rel_l2(full.point_heuristic, ref.point_heuristic) < 10 * GRAD_REL_L2
  assert rel_l2(heur, ref.point_heuristic) > 100 * GRAD_REL_L2, "the sliced sum should not match"


def test_render_gaussians_depth_254_features(cuda_device):
  """render_depth with 254 features: 256 rasterized channels [depth, depth^2, features]"""
  cfg = RasterConfig(compute_visibility=True, compute_point_heuristic=True)
  g, cam = scene3d(5, 3000, image_size=(160, 120), scale_factor=0.5, channels=254)
  gd, cd = g.to(device=cuda_device), cam.to(device=cuda_device)
  gd.requires_grad_(True)
  out = render_gaussians(gd, cd, cfg, use_sh=False, render_depth=True)
  ref, _, _, gr, (img32, w32, vis32) = oracle_render(g, cam, cfg, False, True, out)
  assert out.image.shape == (120, 160, 254)
  assert rel_l2(out.image, img32[..., 2:]) < IMAGE_REL_L2
  assert rel_l2(out.image_weight, w32) < IMAGE_REL_L2
  assert rel_l2(out.point_visibility, vis32) < GRAD_REL_L2
  assert rel_l2(out.image, ref.image[..., 2:]) < 1e-4     # f32 path vs the float64 pipeline
  d_ref = img32[..., 0] / (w32 + 1e-6)
  assert rel_l2(out.depth, d_ref) < IMAGE_REL_L2

  torch.manual_seed(1)
  gi = torch.rand_like(ref.image[..., 2:])
  (out.image * gi.to(cuda_device)).sum().backward()
  (ref.image[..., 2:] * gi.double()).sum().backward()
  errs = {n: rel_l2(getattr(gd, n).grad, getattr(gr, n).grad) for n in ("position", "alpha_logit", "feature")}
  # same bounds as test_render_gaussians_vs_oracle (position goes through the f32 projection)
  assert errs["feature"] < GRAD_REL_L2 and errs["alpha_logit"] < GRAD_REL_L2, errs
  assert errs["position"] < 5e-3, errs


def test_captured_step_256_channels(cuda_device):
  """forward + backward with 256 channels through overlap_capacity= in a CapturedStep: replay equals eager"""
  cfg = RasterConfig(compute_visibility=True, compute_point_heuristic=True)
  g, cam = scene3d(6, 4000, image_size=(160, 120), scale_factor=0.5, channels=256)
  g, cam = g.to(device=cuda_device), cam.to(device=cuda_device)
  g.requires_grad_(True)
  names = ("position", "log_scaling", "rotation", "alpha_logit", "feature")
  params = [getattr(g, n) for n in names]
  torch.manual_seed(2)
  gi = torch.rand(120, 160, 256, device=cuda_device) - 0.3
  static_grads = [torch.zeros_like(p) for p in params]
  holder = {}

  def body():
    for p, b in zip(params, static_grads):
      b.zero_()
      p.grad = b
    out = render_gaussians(g, cam, cfg, use_sh=False, overlap_capacity=300_000)
    (out.image * gi).sum().backward()
    holder["image"] = out.image

  step = CapturedStep(body, device=cuda_device)
  step.replay()
  torch.cuda.synchronize()
  got_image = holder["image"].clone()
  got = [b.clone() for b in static_grads]

  for p in params:
    p.grad = None
  out = render_gaussians(g, cam, cfg, use_sh=False)
  (out.image * gi).sum().backward()
  assert torch.equal(got_image, out.image)
  for n, b, p in zip(names, got, params):
    assert rel_l2(b, p.grad) < 2e-6, (n, rel_l2(b, p.grad))


@pytest.mark.parametrize("channels,antialias,message", [(257, False, "256"), (100, True, "256")])
def test_xwide_limits(cuda_device, channels, antialias, message):
  cfg = RasterConfig(antialias=antialias)
  g, depth, feat = scene2d(3, 200, (64, 48), channels=channels)
  o2p, ranges = oracle.map_to_tiles(g, depth, (64, 48), cfg)
  with pytest.raises(RuntimeError, match=message):
    rasterize_with_tiles(g.to(cuda_device), feat.to(cuda_device), o2p.to(cuda_device), ranges.view(-1, 2).to(cuda_device),
                         (64, 48), cfg)
