"""Differentiable tile rasterizer.

Operator surface of taichi_splatting/rasterizer/function.py: ``rasterize_with_tiles`` (:96-127),
``rasterize`` (:129-161) and ``RasterOut`` (:18-23), same autograd conventions (:41-91): image is
differentiable w.r.t. gaussians2d and features; image_weight, visibility and point_heuristic are
not; point_heuristic is returned zero-filled by forward and filled in place by backward.
Extension: with ``RasterConfig.differentiable_weight`` (alpha blending only) image_weight is differentiable too.
Extension: bfloat16 features with float32 gaussians2d.  The image is bfloat16 (the f32 blend rounded once),
image_weight, visibility and point_heuristic stay float32.  8..256 channels with tile_size 16, alpha blending and no
antialiasing run on bf16 kernels (half the feature, image and image-gradient bytes); any other configuration renders
``features.float()`` and rounds the image, which is what the caller would get doing that cast.
The kernels are csrc/raster_fast_*.cu (f32 / blending / tile 16) and csrc/raster_generic.cu.

Two knobs the reference does not have (module level, defaults give reference parity):
  emulate_stale_tail            reproduce the reference's re-read of stale shared-memory slots in the
                                last group of tiles with more than tile_size^2 overlaps (forward.py:88)
  forward_exit_transmittance    0.0: the forward pass only skips work that cannot change any output
                                (transmittance exactly 0); > 0 trades exactness for an earlier exit
"""
import ctypes
from numbers import Integral

import torch
from beartype import beartype
from beartype.typing import NamedTuple, Optional, Tuple

from .. import _native as N
from ..data_types import RasterConfig
from ..mapper.tile_mapper import map_to_tiles

RasterOut = NamedTuple('RasterOut', [
  ('image', torch.Tensor),
  ('image_weight', torch.Tensor),
  ('point_heuristic', Optional[torch.Tensor]),
  ('visibility', Optional[torch.Tensor])
])

_options = dict(emulate_stale_tail=True, forward_exit_transmittance=0.0)


def set_raster_options(emulate_stale_tail: Optional[bool] = None,
                       forward_exit_transmittance: Optional[float] = None):
  if emulate_stale_tail is not None:
    _options['emulate_stale_tail'] = bool(emulate_stale_tail)
  if forward_exit_transmittance is not None:
    _options['forward_exit_transmittance'] = float(forward_exit_transmittance)
  return dict(_options)


def _raster_params(config: RasterConfig, dtype, image_size, F, V, K, pts_grad, feat_grad):
  return N.GsRasterParams(
    dtype=N.dtype_code(dtype, raster=True), image_width=int(image_size[0]), image_height=int(image_size[1]),
    tile_size=config.tile_size, num_features=F, antialias=int(config.antialias),
    use_alpha_blending=int(config.use_alpha_blending), compute_visibility=int(config.compute_visibility),
    compute_point_heuristic=int(config.compute_point_heuristic), points_requires_grad=int(pts_grad),
    features_requires_grad=int(feat_grad), emulate_stale_tail=int(_options['emulate_stale_tail']),
    pixel_stride_x=config.pixel_stride[0], pixel_stride_y=config.pixel_stride[1], workspace_holds_packed=0,
    kernel_variant=0, num_points=V, num_overlaps=K, clamp_max_alpha=config.clamp_max_alpha,
    alpha_threshold=config.alpha_threshold, saturate_threshold=config.saturate_threshold,
    forward_exit_transmittance=_options['forward_exit_transmittance'])


class _RasterFunction(torch.autograd.Function):

  @staticmethod
  def forward(ctx, gaussians, features, overlap_to_point, tile_overlap_ranges, image_size, config):
    dtype, device = gaussians.dtype, gaussians.device
    V, F = features.shape
    K = overlap_to_point.shape[0]
    w, h = int(image_size[0]), int(image_size[1])
    image_feature = torch.empty((h, w, F), dtype=features.dtype, device=device)   # bf16 features: a bf16 image
    image_alpha = torch.empty((h, w), dtype=dtype, device=device)

    if config.compute_point_heuristic:
      point_heuristic = torch.zeros((V, 2), dtype=dtype, device=device)
    else:
      point_heuristic = torch.empty((0, 2), dtype=dtype, device=device)
    if config.compute_visibility:
      visibility = torch.empty((V,), dtype=dtype, device=device)   # zeroed by the callee
    else:
      visibility = torch.empty((0,), dtype=dtype, device=device)

    params = _raster_params(config, features.dtype, image_size, F, V, K, ctx.needs_input_grad[0],
                            ctx.needs_input_grad[1])
    lib = N.lib()
    ws = N.workspace(lib.gs_raster_workspace_bytes(ctypes.byref(params)), device)
    N.call("gs_raster_fwd", ctypes.byref(params), N.ptr(gaussians), N.ptr(features), N.ptr(tile_overlap_ranges), N.ptr(overlap_to_point),
      N.ptr(image_feature), N.ptr(image_alpha), N.ptr(visibility) if config.compute_visibility else N.ptr(None),
      N.ptr(ws), ctypes.c_size_t(ws.numel()), N.stream_ptr(device))

    ctx.params = params
    ctx.workspace = ws            # packed records are reused by backward
    ctx.overlap_to_point = overlap_to_point
    ctx.tile_overlap_ranges = tile_overlap_ranges
    ctx.point_heuristic = point_heuristic
    ctx.config = config
    if config.differentiable_weight and config.use_alpha_blending:
      ctx.mark_non_differentiable(visibility, point_heuristic)
      ctx.save_for_backward(gaussians, features, image_feature, image_alpha)
    else:
      ctx.mark_non_differentiable(image_alpha, visibility, point_heuristic)
      ctx.save_for_backward(gaussians, features, image_feature)
    ctx.set_materialize_grads(False)   # no zero fills for the non-differentiable outputs' gradients
    return image_feature, image_alpha, point_heuristic, visibility

  @staticmethod
  def backward(ctx, grad_image_feature, grad_alpha, grad_point_heuristic, grad_visibility):
    gaussians, features, image_feature = ctx.saved_tensors[:3]
    need_g, need_f = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
    if grad_image_feature is None:
      grad_image_feature = torch.zeros_like(image_feature)
    grad_gaussians = torch.empty_like(gaussians) if need_g else None   # zeroed by the callee
    # bf16 features: the kernels accumulate an f32 gradient, rounded to the features' dtype for autograd below
    grad_features = torch.empty(features.shape, dtype=gaussians.dtype, device=features.device) if need_f else None
    params = ctx.params
    params.points_requires_grad = int(need_g)
    params.features_requires_grad = int(need_f)
    params.workspace_holds_packed = 1
    heur = ctx.point_heuristic if ctx.config.compute_point_heuristic else None
    if grad_alpha is None:
      N.call("gs_raster_bwd", ctypes.byref(params), N.ptr(gaussians), N.ptr(features), N.ptr(ctx.tile_overlap_ranges),
        N.ptr(ctx.overlap_to_point), N.ptr(image_feature), N.ptr(grad_image_feature.contiguous()),
        N.ptr(grad_gaussians), N.ptr(grad_features), N.ptr(heur), N.ptr(ctx.workspace),
        ctypes.c_size_t(ctx.workspace.numel()), N.stream_ptr(gaussians.device))
    else:   # differentiable_weight: image_alpha was saved as the fourth tensor
      N.call("gs_raster_bwd_with_weight", ctypes.byref(params), N.ptr(gaussians), N.ptr(features),
        N.ptr(ctx.tile_overlap_ranges), N.ptr(ctx.overlap_to_point), N.ptr(image_feature),
        N.ptr(grad_image_feature.contiguous()), N.ptr(ctx.saved_tensors[3]), N.ptr(grad_alpha.contiguous()),
        N.ptr(grad_gaussians), N.ptr(grad_features), N.ptr(heur), N.ptr(ctx.workspace),
        ctypes.c_size_t(ctx.workspace.numel()), N.stream_ptr(gaussians.device))
    if grad_features is not None and grad_features.dtype != features.dtype:
      grad_features = grad_features.to(features.dtype)
    return grad_gaussians, grad_features, None, None, None, None


@beartype
def rasterize_with_tiles(gaussians2d: torch.Tensor, features: torch.Tensor,
                         overlap_to_point: torch.Tensor, tile_overlap_ranges: torch.Tensor,
                         image_size: Tuple[Integral, Integral], config: RasterConfig) -> RasterOut:
  """
  Rasterize an image given 2d gaussians, features and tile overlap information.
  Consider using rasterize instead to also compute tile overlap information.

  Parameters:
      gaussians2d: (N, 7)  packed gaussians (mean, axis, sigma, alpha)
      features: (N, F)   features
      overlap_to_point: (K, ) int32, maps overlap index to point index
      tile_overlap_ranges: (TH * TW, 2) int32, maps tile index to its range of overlap indices
      image_size: (2, ) tuple of ints, (width, height)
      config: RasterConfig

  Returns:
      RasterOut(image (H, W, F), image_weight (H, W), point_heuristic (N, 2), visibility (N,));
      image_weight is differentiable when config.differentiable_weight is set (alpha blending only)
  """
  assert gaussians2d.ndim == 2 and gaussians2d.shape[1] == 7, f"gaussians2d must be Nx7, got {gaussians2d.shape}"
  N.require_cuda(gaussians2d, features, overlap_to_point, tile_overlap_ranges)
  assert features.ndim == 2 and features.shape[0] == gaussians2d.shape[0], \
    f"features must be NxF, got {features.shape} for {gaussians2d.shape[0]} gaussians"
  bf16 = features.dtype == torch.bfloat16
  if bf16 and gaussians2d.dtype != torch.float32:
    raise TypeError(f"bfloat16 features need float32 gaussians2d, got {gaussians2d.dtype}")
  if features.dtype == torch.float16:
    raise TypeError("float16 features are not supported: use bfloat16 (with float32 gaussians2d) or float32")
  assert bf16 or features.dtype == gaussians2d.dtype, f"dtype mismatch {features.dtype} != {gaussians2d.dtype}"
  assert overlap_to_point.dtype == torch.int32 and tile_overlap_ranges.dtype == torch.int32
  ranges = tile_overlap_ranges.reshape(-1, 2).contiguous()
  th = -(-int(image_size[1]) // config.tile_size)
  tw = -(-int(image_size[0]) // config.tile_size)
  assert ranges.shape[0] == th * tw, f"expected {th * tw} tile ranges for image {tuple(image_size)}, got {ranges.shape[0]}"

  upcast = bf16 and not bf16_native(features.shape[1], config)
  image, image_weight, point_heuristic, visibility = _RasterFunction.apply(
    gaussians2d.contiguous(), (features.float() if upcast else features).contiguous(), overlap_to_point.contiguous(),
    ranges, image_size, config)
  if upcast:
    image = image.to(torch.bfloat16)
  return RasterOut(image, image_weight, point_heuristic, visibility)


def bf16_native(num_features: int, config: RasterConfig) -> bool:
  """Whether bfloat16 features of this width and config run on the bf16 kernels (GS_BF16); otherwise they are rendered
  as float32 and the image is rounded.  More than 256 channels go to the kernels too, which reject them."""
  return num_features >= 8 and config.tile_size == 16 and config.use_alpha_blending and not config.antialias


def rasterize(gaussians2d: torch.Tensor, depth: torch.Tensor,
              features: torch.Tensor, image_size: Tuple[Integral, Integral],
              config: RasterConfig, use_depth16: bool = False,
              overlap_capacity: Optional[int] = None,
              overlap_total_out: Optional[torch.Tensor] = None) -> RasterOut:
  """
  Rasterize an image given 2d gaussians, depths and features (tile mapping + rasterization).

  Parameters:
      gaussians2d: (N, 7)  packed gaussians
      depth: (N, 1)   depths (sort key, front to back)
      features: (N, F)   features
      image_size: (2, ) tuple of ints, (width, height)
      config: RasterConfig
      overlap_capacity, overlap_total_out: (extension) see map_to_tiles — bound the overlap count so that nothing
        is read back to the host and the call can sit inside a CUDA graph (benchmarks/configs.py c1_graph)
  """
  assert gaussians2d.shape[0] == depth.shape[0] == features.shape[0], \
    f"Size mismatch: got {gaussians2d.shape}, {depth.shape}, {features.shape}"

  overlap_to_point, tile_overlap_ranges = map_to_tiles(
    gaussians2d, depth, image_size=image_size, config=config, use_depth16=use_depth16,
    overlap_capacity=overlap_capacity, overlap_total_out=overlap_total_out)

  return rasterize_with_tiles(
    gaussians2d, features,
    tile_overlap_ranges=tile_overlap_ranges.view(-1, 2),
    overlap_to_point=overlap_to_point,
    image_size=image_size,
    config=config)
