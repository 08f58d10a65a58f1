"""bfloat16 feature fields (GS_BF16): features, image and image gradient stored in bf16, arithmetic and the geometry in
f32.  The reference for most checks is the f32 path fed the same bf16-representable inputs (bf16 values, upcast): the
forward blends in the same f32 order, so its image is the f32 image rounded once; the backward forms the same sums from
the same (rounded) image.  End to end the float64 oracle bounds what bf16 storage costs."""
import ctypes
import dataclasses

import pytest
import torch

import oracle
from taichi_gaussian_rasterizer_b200 import CapturedStep, RasterConfig, rasterize_with_tiles, render_gaussians
from taichi_gaussian_rasterizer_b200 import _native as N
from taichi_gaussian_rasterizer_b200.rasterizer.function import _raster_params
from util import GRAD_REL_L2, rel_l2, scene2d, scene3d

BF16 = torch.bfloat16
# against the float64 oracle (bf16 unit roundoff 2^-9): about twice the largest value measured over the cases of
# test_vs_float64_oracle on a B200 (image 1.73e-3, gradients 1.67e-3; DESIGN.md §3)
ORACLE_IMAGE_REL_L2 = 3.5e-3
ORACLE_GRAD_REL_L2 = 3.5e-3


def bf16_scene(seed, n, size, channels, scale, cfg):
  g, depth, feat = scene2d(seed, n, size, channels=channels, scale_factor=scale)
  o2p, ranges = oracle.map_to_tiles(g, depth, size, cfg)
  torch.manual_seed(seed + 1)
  grad_image = (torch.rand(size[1], size[0], channels) - 0.3).to(BF16)   # bf16 values, as a bf16 loss would give
  return g, feat.to(BF16), o2p, ranges.view(-1, 2), grad_image


def within_one_ulp(a, b):
  """bf16 tensors equal up to one unit in the last place (the f32 sums behind them are accumulated with atomics in
  no fixed order, so a value sitting on a rounding boundary may round either way)"""
  a, b = a.float(), b.float()
  ulp = torch.maximum(a.abs(), b.abs()) * 2.0 ** -7 + 1e-38
  return bool(((a - b).abs() <= ulp).all())


@pytest.mark.gpu
@pytest.mark.parametrize("channels", [8, 16, 34, 64, 65, 100, 128, 256])
@pytest.mark.parametrize("stats", [False, True])
def test_forward_equals_rounded_f32(cuda_device, channels, stats):
  cfg = RasterConfig(compute_visibility=stats, compute_point_heuristic=stats)
  size = (160, 112)
  g, feat, o2p, ranges, _ = bf16_scene(100 + channels, 1500, size, channels, 2.0, cfg)
  args = (o2p.to(cuda_device), ranges.to(cuda_device), size, cfg)
  out = rasterize_with_tiles(g.to(cuda_device), feat.to(cuda_device), *args)
  ref = rasterize_with_tiles(g.to(cuda_device), feat.float().to(cuda_device), *args)
  assert out.image.dtype == BF16 and out.image_weight.dtype == torch.float32
  assert torch.equal(out.image, ref.image.to(BF16))
  assert torch.equal(out.image_weight, ref.image_weight)
  if stats:   # per tile sums committed with float atomics: equal up to their order
    assert out.visibility.dtype == torch.float32 and rel_l2(out.visibility, ref.visibility) < 1e-6


def abi_backward(cuda_device, g, feat, o2p, ranges, size, cfg, image, grad_image, weight=None, grad_weight=None):
  """gs_raster_bwd(_with_weight) called directly (fresh workspace, packed by the call): f32 gradients of the
  gaussians and features, point heuristic"""
  V, F = feat.shape
  p = _raster_params(cfg, feat.dtype, size, F, V, o2p.shape[0], True, True)
  ws = N.workspace(N.lib().gs_raster_workspace_bytes(ctypes.byref(p)), cuda_device)
  gg = torch.empty((V, 7), device=cuda_device)
  gf = torch.empty((V, F), device=cuda_device)
  heur = torch.zeros((V, 2), device=cuda_device)
  common = (ctypes.byref(p), N.ptr(g), N.ptr(feat), N.ptr(ranges), N.ptr(o2p), N.ptr(image), N.ptr(grad_image))
  tail = (N.ptr(gg), N.ptr(gf), N.ptr(heur), N.ptr(ws), ctypes.c_size_t(ws.numel()), N.stream_ptr(cuda_device))
  if grad_weight is None:
    N.call("gs_raster_bwd", *common, *tail)
  else:
    N.call("gs_raster_bwd_with_weight", *common, N.ptr(weight), N.ptr(grad_weight), *tail)
  return gg, gf, heur


@pytest.mark.gpu
@pytest.mark.parametrize("channels", [8, 34, 64, 100, 256])
@pytest.mark.parametrize("with_weight", [False, True])
def test_abi_backward_vs_f32(cuda_device, channels, with_weight):
  cfg = RasterConfig(compute_visibility=True, compute_point_heuristic=True)
  size = (160, 112)
  g, feat, o2p, ranges, grad_image = bf16_scene(200 + channels, 1500, size, channels, 2.0, cfg)
  g, feat, o2p, ranges = g.to(cuda_device), feat.to(cuda_device), o2p.to(cuda_device), ranges.to(cuda_device)
  grad_image = grad_image.to(cuda_device)
  out = rasterize_with_tiles(g, feat, o2p, ranges, size, cfg)
  weight = out.image_weight
  torch.manual_seed(channels)
  grad_weight = (torch.rand(size[1], size[0], device=cuda_device) - 0.5) if with_weight else None
  got = abi_backward(cuda_device, g, feat, o2p, ranges, size, cfg, out.image, grad_image, weight, grad_weight)
  ref = abi_backward(cuda_device, g, feat.float(), o2p, ranges, size, cfg, out.image.float(), grad_image.float(),
                     weight, grad_weight)
  for name, a, b in zip(("grad_gaussians", "grad_features", "point_heuristic"), got, ref):
    assert a.dtype == torch.float32
    assert rel_l2(a, b) < GRAD_REL_L2, (name, rel_l2(a, b))


def autograd_vs_abi(cuda_device, seed, n, size, channels, scale, cfg):
  g, feat, o2p, ranges, grad_image = bf16_scene(seed, n, size, channels, scale, cfg)
  g, o2p, ranges, grad_image = g.to(cuda_device), o2p.to(cuda_device), ranges.to(cuda_device), grad_image.to(cuda_device)
  gd, fd = g.clone().requires_grad_(True), feat.to(cuda_device).requires_grad_(True)
  out = rasterize_with_tiles(gd, fd, o2p, ranges, size, cfg)
  (out.image * grad_image).sum().backward()
  assert fd.grad.dtype == BF16 and gd.grad.dtype == torch.float32
  gg, gf, heur = abi_backward(cuda_device, g, fd.detach(), o2p, ranges, size, cfg, out.image.detach(), grad_image)
  assert within_one_ulp(fd.grad, gf.to(BF16))
  assert rel_l2(gd.grad, gg) < 1e-6
  if cfg.compute_point_heuristic:
    assert rel_l2(out.point_heuristic, heur) < 1e-6
  return out


@pytest.mark.gpu
@pytest.mark.parametrize("channels", [16, 40, 128])
def test_autograd_equals_abi(cuda_device, channels):
  cfg = RasterConfig(compute_visibility=True, compute_point_heuristic=True)
  autograd_vs_abi(cuda_device, 300 + channels, 1500, (160, 112), channels, 2.0, cfg)


@pytest.mark.gpu
def test_autograd_multi_group_tile(cuda_device):
  """tiles with several hundred overlaps (many staged batches, saturation exits)"""
  cfg = RasterConfig(compute_visibility=True, compute_point_heuristic=True)
  autograd_vs_abi(cuda_device, 78, 3000, (64, 48), 130, 6.0, cfg)


@pytest.mark.gpu
def test_autograd_pixel_stride(cuda_device):
  cfg = RasterConfig(pixel_stride=(2, 2), compute_visibility=True, compute_point_heuristic=True)
  autograd_vs_abi(cuda_device, 79, 1500, (160, 112), 200, 2.0, cfg)


@pytest.mark.gpu
@pytest.mark.parametrize("channels", [8, 34, 100, 256])
def test_vs_float64_oracle(cuda_device, channels):
  """what bf16 storage costs end to end: the bf16 image and the rounded feature gradient against the float64 oracle
  of the same (bf16-valued) inputs"""
  cfg = RasterConfig(compute_visibility=True, compute_point_heuristic=True)
  size = (160, 112)
  g, feat, o2p, ranges, grad_image = bf16_scene(400 + channels, 1500, size, channels, 2.0, cfg)
  gr, fr = g.double().requires_grad_(True), feat.double().requires_grad_(True)
  ref = oracle.rasterize_with_tiles(gr, fr, o2p, ranges, size, cfg)
  (ref.image * grad_image.double()).sum().backward()
  gd, fd = g.to(cuda_device).requires_grad_(True), feat.to(cuda_device).requires_grad_(True)
  out = rasterize_with_tiles(gd, fd, o2p.to(cuda_device), ranges.to(cuda_device), size, cfg)
  (out.image * grad_image.to(cuda_device)).sum().backward()
  errs = dict(image=rel_l2(out.image.double(), ref.image), grad_gaussians=rel_l2(gd.grad.double(), gr.grad),
              grad_features=rel_l2(fd.grad.double(), fr.grad))
  print(f"bf16 vs float64 oracle, F={channels}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
  assert errs["image"] < ORACLE_IMAGE_REL_L2, errs
  assert errs["grad_gaussians"] < ORACLE_GRAD_REL_L2 and errs["grad_features"] < ORACLE_GRAD_REL_L2, errs


def with_feature(g, feature):
  return dataclasses.replace(g, feature=feature)


@pytest.mark.gpu
def test_render_gaussians_bf16(cuda_device):
  cfg = RasterConfig(compute_visibility=True, compute_point_heuristic=True)
  g, cam = scene3d(5, 3000, image_size=(160, 120), scale_factor=0.5, channels=128)
  g, cam = g.to(device=cuda_device), cam.to(device=cuda_device)
  gb = with_feature(g, g.feature.to(BF16)).requires_grad_(True)
  gf = with_feature(g, gb.feature.detach().float()).requires_grad_(True)
  out = render_gaussians(gb, cam, cfg, use_sh=False)
  ref = render_gaussians(gf, cam, cfg, use_sh=False)
  assert out.image.dtype == BF16 and out.image_weight.dtype == torch.float32
  assert torch.equal(out.image, ref.image.to(BF16))
  torch.manual_seed(1)
  gi = (torch.rand(120, 160, 128, device=cuda_device) - 0.3).to(BF16)
  (out.image * gi).sum().backward()
  (ref.image * gi.float()).sum().backward()
  assert gb.feature.grad.dtype == BF16
  errs = {n: rel_l2(getattr(gb, n).grad.float(), getattr(gf, n).grad) for n in ("position", "alpha_logit", "feature")}
  print(f"render_gaussians bf16 vs f32 gradients: {errs}")
  assert all(e < ORACLE_GRAD_REL_L2 for e in errs.values()), errs


@pytest.mark.gpu
@pytest.mark.parametrize("static", [False, True])
def test_render_depth_bf16(cuda_device, static):
  """render_depth widens the visible rows to f32 behind the depth channels: depth and depth_var are the f32 path's"""
  cfg = RasterConfig()
  g, cam = scene3d(7, 3000, image_size=(160, 120), scale_factor=0.5, channels=32)
  g, cam = g.to(device=cuda_device), cam.to(device=cuda_device)
  gb = with_feature(g, g.feature.to(BF16))
  gf = with_feature(g, gb.feature.float())
  kw = dict(use_sh=False, render_depth=True, overlap_capacity=200_000 if static else None)
  out, ref = render_gaussians(gb, cam, cfg, **kw), render_gaussians(gf, cam, cfg, **kw)
  assert out.image.dtype == BF16 and out.depth.dtype == torch.float32 and out.depth_var.dtype == torch.float32
  assert torch.equal(out.depth, ref.depth) and torch.equal(out.depth_var, ref.depth_var)
  assert torch.equal(out.image, ref.image.to(BF16))


@pytest.mark.gpu
def test_captured_step_256_channels_bf16(cuda_device):
  """forward + backward with 256 bf16 channels through overlap_capacity= in a CapturedStep: replay equals eager"""
  cfg = RasterConfig(compute_visibility=True, compute_point_heuristic=True)
  g, cam = scene3d(6, 4000, image_size=(160, 120), scale_factor=0.5, channels=256)
  g, cam = g.to(device=cuda_device), cam.to(device=cuda_device)
  g = with_feature(g, g.feature.to(BF16)).requires_grad_(True)
  names = ("position", "log_scaling", "rotation", "alpha_logit", "feature")
  params = [getattr(g, n) for n in names]
  torch.manual_seed(2)
  gi = (torch.rand(120, 160, 256, device=cuda_device) - 0.3).to(BF16)
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
  assert out.image.dtype == BF16 and torch.equal(got_image, out.image)
  for n, b, p in zip(names, got, params):
    if n == "feature":   # bf16: the f32 sums behind it may round either way where they sit on a boundary
      assert b.dtype == BF16 and within_one_ulp(b, p.grad), n
    else:
      assert rel_l2(b, p.grad) < 2e-6, (n, rel_l2(b, p.grad))


@pytest.mark.gpu
@pytest.mark.parametrize("channels,cfg", [(3, RasterConfig()), (16, RasterConfig(antialias=True)),
                                          (16, RasterConfig(tile_size=8, pixel_stride=(1, 1)))])
def test_upcast_path(cuda_device, channels, cfg):
  """no bf16 kernel for these: the f32 path on features.float(), the image rounded to bf16 — as the caller's cast"""
  size = (96, 64)
  g, feat, o2p, ranges, grad_image = bf16_scene(500 + channels, 800, size, channels, 1.5, cfg)
  args = (o2p.to(cuda_device), ranges.to(cuda_device), size, cfg)
  fd = feat.to(cuda_device).requires_grad_(True)
  out = rasterize_with_tiles(g.to(cuda_device), fd, *args)
  ref = rasterize_with_tiles(g.to(cuda_device), fd.detach().float(), *args)
  assert out.image.dtype == BF16 and torch.equal(out.image, ref.image.to(BF16))
  (out.image * grad_image.to(cuda_device)).sum().backward()
  assert fd.grad.dtype == BF16


@pytest.mark.gpu
def test_errors(cuda_device):
  cfg = RasterConfig()
  size = (64, 48)
  g, feat, o2p, ranges, _ = bf16_scene(3, 200, size, 16, 1.0, cfg)
  args = (o2p.to(cuda_device), ranges.to(cuda_device), size, cfg)
  with pytest.raises(TypeError, match="float32 gaussians2d"):
    rasterize_with_tiles(g.double().to(cuda_device), feat.to(cuda_device), *args)
  with pytest.raises(TypeError, match="float16 features"):
    rasterize_with_tiles(g.to(cuda_device), feat.half().to(cuda_device), *args)
  g, feat, o2p, ranges, _ = bf16_scene(3, 200, size, 257, 1.0, cfg)
  with pytest.raises(RuntimeError, match="256"):
    rasterize_with_tiles(g.to(cuda_device), feat.to(cuda_device), o2p.to(cuda_device), ranges.to(cuda_device), size,
                         cfg)


def bf16_params(**kw):
  base = dict(dtype=N.GS_BF16, image_width=64, image_height=48, tile_size=16, num_features=32, antialias=0,
              use_alpha_blending=1, pixel_stride_x=1, pixel_stride_y=1, num_points=1000, num_overlaps=5000)
  base.update(kw)
  return N.GsRasterParams(**base)


@pytest.mark.parametrize("kw,message", [(dict(num_features=4), b"8..256"), (dict(num_features=257), b"256"),
                                        (dict(antialias=1), b"antialiasing"), (dict(tile_size=8), b"tile_size 16"),
                                        (dict(use_alpha_blending=0), b"alpha blending")])
def test_abi_rejects_bf16_without_kernels(kw, message):
  lib = N.lib()
  p = bf16_params(**kw)
  rc = lib.gs_raster_fwd(ctypes.byref(p), None, None, None, None, None, None, None, None, ctypes.c_size_t(0), None)
  assert rc == -2 and message in lib.gs_last_error_string()
  rc = lib.gs_raster_bwd(ctypes.byref(p), None, None, None, None, None, None, None, None, None, None,
                         ctypes.c_size_t(0), None)
  assert rc == -2 and message in lib.gs_last_error_string()


@pytest.mark.parametrize("channels", [8, 34, 100, 128, 256])
def test_bf16_workspace_is_smaller(channels):
  lib = N.lib()
  bf = lib.gs_raster_workspace_bytes(ctypes.byref(bf16_params(num_features=channels)))
  f32 = lib.gs_raster_workspace_bytes(ctypes.byref(bf16_params(num_features=channels, dtype=N.GS_F32)))
  assert 0 < bf <= f32
  if channels not in (128, 256):   # rows read in place in both: the workspace holds records and cull bytes only
    assert bf < f32
