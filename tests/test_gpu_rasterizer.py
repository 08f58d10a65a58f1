"""Rasterizer forward / backward on the GPU against the oracle (north_star tolerances: images 1e-5,
gradients 1e-4 relative L2 in fp32), plus the reference's own checks re-hosted on the CUDA kernels:
float64 gradcheck of the single tile setup (tests/test_rasterizer.py:30-90) and visibility == feature
gradient (tests/test_visibility.py:34-63)."""
import pytest
import torch

import oracle
from taichi_gaussian_rasterizer_b200 import RasterConfig, rasterize, rasterize_with_tiles, set_raster_options
from util import GRAD_REL_L2, IMAGE_REL_L2, rel_l2, scene2d

pytestmark = pytest.mark.gpu


def compare_forward_backward(cuda_device, seed, n, size, cfg, channels=3, scale=1.0, alpha_range=(0.1, 0.9),
                             dtype=torch.float32, check_grads=True):
  g, depth, feat = scene2d(seed, n, size, channels=channels, scale_factor=scale, alpha_range=alpha_range, dtype=dtype)
  o2p, ranges = oracle.map_to_tiles(g.float(), depth, size, cfg)
  torch.manual_seed(seed + 1)
  grad_image = torch.rand(size[1], size[0], channels, dtype=dtype) - 0.3

  gr, fr = g.clone().requires_grad_(True), feat.clone().requires_grad_(True)
  ref = oracle.rasterize_with_tiles(gr, fr, o2p, ranges.view(-1, 2), size, cfg)
  gd, fd = g.to(cuda_device).requires_grad_(True), feat.to(cuda_device).requires_grad_(True)
  out = rasterize_with_tiles(gd, fd, o2p.to(cuda_device), ranges.view(-1, 2).to(cuda_device), size, cfg)

  assert out.image.shape == ref.image.shape and out.image_weight.shape == ref.image_weight.shape
  assert rel_l2(out.image, ref.image) < IMAGE_REL_L2, f"image rel l2 {rel_l2(out.image, ref.image)}"
  assert rel_l2(out.image_weight, ref.image_weight) < IMAGE_REL_L2
  if cfg.compute_visibility:
    assert rel_l2(out.visibility, ref.visibility) < GRAD_REL_L2
  else:
    assert out.visibility.shape == (0,)
  if check_grads:
    (ref.image * grad_image).sum().backward()
    (out.image * grad_image.to(cuda_device)).sum().backward()
    assert rel_l2(gd.grad, gr.grad) < GRAD_REL_L2, f"gaussian grad rel l2 {rel_l2(gd.grad, gr.grad)}"
    assert rel_l2(fd.grad, fr.grad) < GRAD_REL_L2, f"feature grad rel l2 {rel_l2(fd.grad, fr.grad)}"
    if cfg.compute_point_heuristic:
      assert rel_l2(out.point_heuristic, ref.point_heuristic) < 10 * GRAD_REL_L2
    else:
      assert out.point_heuristic.shape == (0, 2)
  return out, ref


@pytest.mark.parametrize("seed,n,size,scale", [(0, 500, (128, 96), 1.0), (1, 3000, (200, 150), 2.0),
                                               (2, 20000, (333, 257), 2.0), (3, 4000, (64, 64), 6.0)])
def test_fast_path_vs_oracle(cuda_device, seed, n, size, scale):
  """f32, blending, tile 16: the measured kernels; (3) has tiles with several hundred to >1000 overlaps."""
  cfg = RasterConfig(compute_visibility=True, compute_point_heuristic=True)
  compare_forward_backward(cuda_device, seed, n, size, cfg, scale=scale)


def test_multi_group_tiles_and_stale_tail(cuda_device):
  """Tiles with C > 256 and C % 256 != 0 exercise the reference's stale-slot re-read (SURVEY Q1);
  low opacities keep pixels unsaturated so the re-read is visible in the image."""
  cfg = RasterConfig()
  size = (48, 32)
  for emulate in (True, False):
    set_raster_options(emulate_stale_tail=emulate)
    try:
      g, depth, feat = scene2d(5, 2500, size, scale_factor=8.0, alpha_range=(0.01, 0.05))
      o2p, ranges = oracle.map_to_tiles(g, depth, size, cfg)
      counts = (ranges[..., 1] - ranges[..., 0]).view(-1)
      assert int(counts.max()) > 256 and any(int(c) % 256 for c in counts)
      ref_img, ref_w, _ = oracle.raster_forward(g, feat, o2p, ranges.view(-1, 2), size, cfg, emulate_stale_tail=emulate)
      out = rasterize_with_tiles(g.to(cuda_device), feat.to(cuda_device), o2p.to(cuda_device),
                                 ranges.view(-1, 2).to(cuda_device), size, cfg)
      assert rel_l2(out.image, ref_img) < IMAGE_REL_L2
      assert rel_l2(out.image_weight, ref_w) < IMAGE_REL_L2
    finally:
      set_raster_options(emulate_stale_tail=True)
  a, _, _ = oracle.raster_forward(g, feat, o2p, ranges.view(-1, 2), size, cfg, emulate_stale_tail=True)
  b, _, _ = oracle.raster_forward(g, feat, o2p, ranges.view(-1, 2), size, cfg, emulate_stale_tail=False)
  assert rel_l2(a, b) > 1e-3, "scene does not exercise the quirk"


@pytest.mark.parametrize("channels", [1, 2, 4, 5, 7, 8])
def test_feature_widths_fast(cuda_device, channels):
  cfg = RasterConfig()
  compare_forward_backward(cuda_device, 10 + channels, 1500, (160, 112), cfg, channels=channels, scale=2.0)


@pytest.mark.parametrize("channels,stats", [(8, False), (8, True), (9, True), (12, False), (16, True), (17, False), (34, False),
                                            (34, True), (36, False), (37, False), (64, True)])
def test_wide_features(cuda_device, channels, stats):
  """8..64 channels take the wide kernels (forward FP 16/36/64, backward one pixel per lane); 34 channels is
  BASELINE.json's feature-lifting configuration (depth, depth^2, 32 features)."""
  cfg = RasterConfig(compute_visibility=stats, compute_point_heuristic=stats)
  # same scene size as test_feature_widths_fast: one alpha_threshold decision that flips between ex2.approx and
  # libm exp moves a pixel by ~0.4 %, which alone is 4e-5 relative L2 of a 96x80 image but 1e-5 of this one
  compare_forward_backward(cuda_device, 20 + channels, 1500, (160, 112), cfg, channels=channels, scale=2.0)


def test_wide_features_multi_group_tile(cuda_device):
  """wide kernels on tiles with several hundred overlaps (many batches, saturation exits)"""
  cfg = RasterConfig()
  compare_forward_backward(cuda_device, 77, 3000, (64, 48), cfg, channels=34, scale=6.0)


@pytest.mark.parametrize("ts,stride", [(8, (1, 1)), (8, (2, 1)), (32, (2, 2)), (32, (4, 4))])
def test_tile_sizes_generic(cuda_device, ts, stride):
  cfg = RasterConfig(tile_size=ts, pixel_stride=stride, compute_visibility=True, compute_point_heuristic=True)
  compare_forward_backward(cuda_device, 30 + ts, 1500, (150, 100), cfg, scale=2.0)


def test_antialias_generic(cuda_device):
  cfg = RasterConfig(antialias=True, blur_cov=0.0, compute_visibility=True)
  compare_forward_backward(cuda_device, 40, 1500, (150, 100), cfg, scale=1.0)


@pytest.mark.parametrize("seed,n,size,scale,channels", [(42, 3000, (200, 150), 1.0, 3), (43, 4000, (64, 64), 6.0, 3),
                                                         (44, 20000, (1024, 1024), 0.5, 3), (45, 1500, (160, 112), 2.0, 5),
                                                         (46, 2000, (100, 70), 0.3, 1)])
def test_antialias_fast_path(cuda_device, seed, n, size, scale, channels):
  """antialias=True at tile 16 with narrow features runs the measured (fast) kernels: the pixel-integrated gaussian
  (taichi_lib/generic.py:340-404) with visibility and split / prune statistics — BASELINE.json config 1's setting
  (examples/fit_image_gaussians.py:289-296); (43) has tiles with many hundred overlaps, (46) sub-pixel gaussians."""
  cfg = RasterConfig(antialias=True, blur_cov=0.0, compute_visibility=True, compute_point_heuristic=True)
  compare_forward_backward(cuda_device, seed, n, size, cfg, channels=channels, scale=scale,
                           alpha_range=(0.5, 1.0) if seed == 44 else (0.1, 0.9))


def test_quantile_mode_forward(cuda_device):
  cfg = RasterConfig(use_alpha_blending=False, saturate_threshold=0.5)
  size = (150, 100)
  g, depth, feat = scene2d(41, 2000, size, channels=1, scale_factor=2.0, alpha_range=(0.3, 0.9))
  o2p, ranges = oracle.map_to_tiles(g, depth, size, cfg)
  ref_img, ref_w, _ = oracle.raster_forward(g, depth.clone(), o2p, ranges.view(-1, 2), size, cfg)
  out = rasterize_with_tiles(g.to(cuda_device), depth.to(cuda_device), o2p.to(cuda_device),
                             ranges.view(-1, 2).to(cuda_device), size, cfg)
  # a selection, not a blend: allow a vanishing number of pixels to pick a neighbouring gaussian
  diff = (out.image.cpu() != ref_img).float().mean().item()
  assert diff < 1e-3
  assert torch.equal(out.image_weight.cpu(), ref_w)


@pytest.mark.parametrize("dtype,tile,antialias", [(torch.float32, 16, False), (torch.float64, 8, False),
                                                  (torch.float32, 16, True)])
def test_quantile_mode_backward(cuda_device, dtype, tile, antialias):
  """SURVEY 8f rank 3: each pixel's image gradient goes to the features of the gaussian the forward selected;
  the packed gaussians get zeros.  Checked against the selection itself (rendered with index features, by the CUDA
  path and by the oracle) — the reference has no backward for this mode (tests/test_rasterizer.py:92-94)."""
  cfg = RasterConfig(use_alpha_blending=False, saturate_threshold=0.5, tile_size=tile, pixel_stride=(1, 1),
                     antialias=antialias, blur_cov=0.0 if antialias else 0.3)
  size = (150, 100)
  g, depth, feat = scene2d(43, 2000, size, channels=2, scale_factor=2.0, alpha_range=(0.3, 0.9), dtype=dtype)
  o2p, ranges = oracle.map_to_tiles(g.float(), depth, size, cfg)
  o2p_d, ranges_d = o2p.to(cuda_device), ranges.view(-1, 2).to(cuda_device)
  V = g.shape[0]
  torch.manual_seed(7)
  grad_image = (torch.rand(size[1], size[0], 2, dtype=dtype) - 0.3).to(cuda_device)

  gd, fd = g.to(cuda_device).requires_grad_(True), feat.to(cuda_device).requires_grad_(True)
  out = rasterize_with_tiles(gd, fd, o2p_d, ranges_d, size, cfg)
  (out.image * grad_image).sum().backward()

  ids = torch.arange(1, V + 1, dtype=dtype).view(-1, 1)
  sel = rasterize_with_tiles(g.to(cuda_device), ids.to(cuda_device), o2p_d, ranges_d, size, cfg).image[..., 0].long()
  hit = sel > 0
  assert hit.float().mean() > 0.5
  expect = torch.zeros(V, 2, dtype=dtype, device=cuda_device).index_add_(0, sel[hit] - 1, grad_image[hit])
  assert torch.allclose(fd.grad, expect, rtol=1e-5, atol=1e-6)
  assert torch.equal(out.image[hit], feat.to(cuda_device)[sel[hit] - 1])
  assert gd.grad is not None and not gd.grad.any()
  # the oracle selects the same gaussians (up to a vanishing number of borderline pixels)
  sel_ref = oracle.raster_forward(g, ids, o2p, ranges.view(-1, 2), size, cfg)[0][..., 0].long()
  assert (sel.cpu() != sel_ref).float().mean().item() < 1e-3


def test_quantile_mode_gradcheck_and_median_depth_gradient(cuda_device):
  """float64 gradcheck of quantile mode w.r.t. the features (the case the reference leaves commented out), and the
  median depth of render_gaussians back-propagating to the gaussian positions."""
  cfg = RasterConfig(tile_size=8, pixel_stride=(1, 1), use_alpha_blending=False, saturate_threshold=0.5)
  size = (24, 16)
  g, depth, feat = scene2d(44, 40, size, channels=2, scale_factor=3.0, alpha_range=(0.4, 0.9), dtype=torch.float64)
  o2p, ranges = oracle.map_to_tiles(g.float(), depth, size, cfg)
  gd, o2p, ranges = g.to(cuda_device), o2p.to(cuda_device), ranges.view(-1, 2).to(cuda_device)
  fd = feat.to(cuda_device).requires_grad_(True)
  assert torch.autograd.gradcheck(lambda f: rasterize_with_tiles(gd, f, o2p, ranges, size, cfg).image, (fd,),
                                  eps=1e-6, nondet_tol=1e-9)

  from taichi_gaussian_rasterizer_b200 import render_gaussians
  from taichi_gaussian_rasterizer_b200.synthetic import random_3d_gaussians, random_camera
  torch.manual_seed(3)
  cam = random_camera(image_size=(96, 64))
  g3 = random_3d_gaussians(800, cam, scale_factor=2.0, alpha_range=(0.5, 0.95)).to(device=cuda_device).requires_grad_(True)
  r = render_gaussians(g3, cam.to(device=cuda_device), RasterConfig(), render_median_depth=True)
  assert r.median_depth.shape == (64, 96) and r.median_depth.requires_grad
  r.median_depth.sum().backward()
  assert g3.position.grad is not None and g3.position.grad.abs().sum() > 0
  covered = (r.median_depth > 0).sum().item()
  # d(sum of median depths)/d(depth_i) = number of pixels that selected gaussian i; total = covered pixels
  assert covered > 0


def test_invalid_pixel_stride_is_rejected(cuda_device):
  cfg = RasterConfig(tile_size=8, pixel_stride=(2, 2))   # 64 / 4 = 16 < 32 threads
  g, depth, feat = scene2d(0, 10, (16, 16))
  with pytest.raises(RuntimeError, match="pixel_stride"):
    rasterize(g.to(cuda_device), depth.to(cuda_device), feat.to(cuda_device), (16, 16), cfg)


def test_empty_inputs(cuda_device):
  cfg = RasterConfig(compute_visibility=True, compute_point_heuristic=True)
  size = (40, 24)
  out = rasterize(torch.zeros((0, 7), device=cuda_device), torch.zeros((0, 1), device=cuda_device),
                  torch.zeros((0, 3), device=cuda_device), size, cfg)
  assert out.image.shape == (24, 40, 3) and float(out.image.abs().sum()) == 0 and float(out.image_weight.sum()) == 0
  assert out.visibility.shape == (0,) and out.point_heuristic.shape == (0, 2)


# ---- the reference's own rasterizer tests, re-hosted -------------------------------------------------------
def make_inputs(config, seed, device):
  torch.manual_seed(seed)
  n = int(torch.randint(1, 50, (1,)))
  channels = int(torch.randint(1, 4, (1,)))
  image_size = (8, 8)
  g, _, feat = scene2d(seed, n, image_size, channels=channels, alpha_range=(0.2, 0.8), dtype=torch.float64)
  g, feat = g.to(device), feat.to(device)
  o2p = torch.arange(0, n, device=device, dtype=torch.int32)
  tile_ranges = torch.tensor([[0, n]], device=device, dtype=torch.int32)

  def render(mean, axis, sigma, alpha, colors):
    packed = torch.cat([mean, axis, sigma, alpha], dim=-1)
    return rasterize_with_tiles(packed, colors, overlap_to_point=o2p, tile_overlap_ranges=tile_ranges.view(-1, 2),
                                image_size=image_size, config=config).image

  return (g[:, 0:2].requires_grad_(True), g[:, 2:4].requires_grad_(True), g[:, 4:6].requires_grad_(True),
          g[:, 6:7].requires_grad_(True), feat.requires_grad_(True)), render


@pytest.mark.parametrize("antialias", [True, False])
def test_rasterizer_gradcheck(cuda_device, antialias):
  config = RasterConfig(tile_size=8, pixel_stride=(1, 1), antialias=antialias, use_alpha_blending=True)
  torch.manual_seed(0)
  seeds = torch.randint(0, 1000, (25,))
  for seed in seeds:
    inputs, render = make_inputs(config, int(seed), cuda_device)
    torch.autograd.gradcheck(render, inputs, eps=1e-6, check_grad_dtypes=True, check_undefined_grad=False,
                             nondet_tol=1e-9)


def test_visibility(cuda_device):
  torch.manual_seed(0)
  image_size = (320, 200)
  config = RasterConfig(compute_visibility=True, compute_point_heuristic=True)
  for i in range(6):
    n = int(torch.randint(1, 10000, (1,)))
    g, depth, feat = scene2d(50 + i, n, image_size, scale_factor=0.2, alpha_range=(0.2, 1.0), dtype=torch.float64)
    feat = feat.to(cuda_device).requires_grad_(True)
    raster = rasterize(gaussians2d=g.to(cuda_device), depth=depth.to(cuda_device), features=feat,
                       image_size=image_size, config=config)
    raster.image.sum().backward()
    assert torch.allclose(feat.grad[:, 0], raster.visibility, rtol=1e-7, atol=1e-10)
    # f32 fast kernels: same relation within fp32 accumulation error
    f32 = feat.detach().float().requires_grad_(True)
    r32 = rasterize(g.float().to(cuda_device), depth.to(cuda_device), f32, image_size, config)
    r32.image.sum().backward()
    assert rel_l2(f32.grad[:, 0], r32.visibility) < GRAD_REL_L2
