"""Complete 3D gaussian renderer: project -> (SH) -> tile map -> rasterize.

Operator surface of taichi_splatting/renderer.py: ``render_gaussians`` (:133-170),
``render_projected`` (:183-231) and ``viewspace_gradient`` (:234-239); the ``Rendering`` result lives in
rendering.py.  The two ``torch.compile`` helpers of the reference (ndc_depth, depth variance) are plain eager
torch here.
"""
from dataclasses import replace
from typing import Optional

import torch
from beartype import beartype

from .data_types import Gaussians3D, RasterConfig
from .mapper.tile_mapper import (_map_to_tiles, launch_mapper_front_counted, map_front_to_tiles_capped,
                                 map_to_tiles)
from .perspective import CameraParams
from .perspective.projection import project_to_image, project_to_image_static
from .rasterizer.function import rasterize_with_tiles
from .rendering import Rendering
from .spherical_harmonics import (evaluate_sh_at, launch_gather_counted, launch_gather_into, launch_sh_forward_counted,
                                  launch_sh_forward_into)
from .torch_lib.projection import ndc_depth


@beartype
def render_gaussians(
  gaussians: Gaussians3D,
  camera_params: CameraParams,
  config: RasterConfig = RasterConfig(),
  use_sh: bool = False,
  render_depth: bool = False,
  use_depth16: bool = False,
  render_median_depth: bool = False,
  sh_colors: Optional[torch.Tensor] = None,
  overlap_capacity: Optional[int] = None,
  overlap_total_out: Optional[torch.Tensor] = None
) -> Rendering:
  """
  A complete renderer for 3D gaussians.
  Parameters:
    gaussians: Gaussians3D - feature is (N, C), or (N, 3, (D+1)**2) spherical harmonics if use_sh
    camera_params: CameraParams
    config: RasterConfig
    use_sh: bool - whether to evaluate spherical harmonics for the view direction
    render_depth: bool - whether to render depth and depth variance
    use_depth16: bool - whether to use 16 bit depth encoding for sorting (otherwise 32 bit)
    render_median_depth: bool - whether to render the median depth map
    sh_colors: (extension) with use_sh, this view's dense (N, 3) colours from ``evaluate_sh_views`` (one pass over the
      SH coefficients for the whole batch of views): the visible rows are gathered instead of evaluated; autograd
      still reaches ``gaussians.feature``
    overlap_capacity: (extension) bound on the number of tile overlaps K.  The call then reads NOTHING back to the
      host (the reference synchronises the device four times per view: torch.nonzero, two cudaDeviceSynchronize in
      cuda_lib, and the size of the key buffers): the visible count V and K stay on the device, the point space
      tensors of the result keep N rows (``points_in_view_count`` holds V), overlaps beyond the capacity are dropped
      (pass a (1,) int32 CUDA tensor as ``overlap_total_out`` to receive K and compare it with the capacity now and
      then).  Same kernels and the same values as the default path; forward + backward of any number of views can be
      captured in ONE CUDA graph (bench.py).  f32 gaussians only.
    bfloat16 plain features (use_sh=False, float32 geometry): the image is bfloat16 and the feature rows stay bf16 from
      the gather to the rasterizer (see rasterizer.function); with render_depth the visible rows are widened to
      float32 behind the f32 depth channels and only the returned image is rounded back to bf16 (depth, depth_var f32).

  Returns:
    Rendering - rendered image, with optional depth / depth variance and per point statistics
  """
  if overlap_capacity is not None:
    return _render_gaussians_static(gaussians, camera_params, config, use_sh, render_depth, use_depth16,
                                    render_median_depth, sh_colors, int(overlap_capacity), overlap_total_out)
  # issued before the projection so that these few tiny launches overlap with it instead of sitting behind the
  # host read-back of the visible count
  camera_position = camera_params.camera_position if use_sh else None
  early = {}
  sh_early = use_sh and gaussians.feature.is_contiguous() and gaussians.position.is_contiguous() \
    and gaussians.position.dtype == gaussians.feature.dtype
  order_early = gaussians.position.dtype == torch.float32
  assert sh_colors is None or sh_early, "sh_colors needs use_sh and contiguous features / positions of one dtype"

  # Work that only needs the device-side visible set is enqueued right behind the projection kernel, BEFORE the host
  # blocks on the visible count: the front half of the tile mapper (depth ordering, overlap count, scan: 0.3 ms at 3 M
  # gaussians), so that the GPU idles neither across that read-back nor during the host's work after it.
  def early_work(indexes_capacity, count_device, depth_capacity, points_capacity):
    early["front"] = launch_mapper_front_counted(points_capacity, depth_capacity, count_device,
                                                 camera_params.image_size, config, use_depth16,
                                                 (camera_params.near_plane, camera_params.far_plane))
  gaussians2d, depths, indexes = project_to_image(gaussians, camera_params, config,
                                                  after_launch=early_work if order_early else None)

  fill_features = None
  depth_in_features = False
  if use_sh and sh_early:
    # The colours do not depend on the tile map: their kernel (the SH evaluation, or the gather of this view's rows of
    # a batch evaluation) is enqueued by the tile mapper right before it waits for the overlap total, to keep the GPU
    # busy across THAT read-back.  The autograd node is built now, around the buffer the kernel will fill.
    pre = torch.empty((indexes.shape[0], gaussians.feature.shape[1]), dtype=gaussians.feature.dtype,
                      device=gaussians.feature.device)
    if sh_colors is not None:
      assert sh_colors.shape == (gaussians.feature.shape[0], gaussians.feature.shape[1]) and sh_colors.is_contiguous()
      fill_features = lambda: launch_gather_into(sh_colors, indexes, pre)   # noqa: E731
    else:
      cam_pos = camera_position.detach().to(gaussians.feature.dtype).contiguous()
      fill_features = lambda: launch_sh_forward_into(gaussians.feature.detach(), gaussians.position.detach(),   # noqa: E731
                                                     indexes, cam_pos, pre)
    features = evaluate_sh_at(gaussians.feature, gaussians.position.detach(), indexes,
                              camera_position, indexes_sorted_unique=True,   # visible set: ascending
                              precomputed=pre)
  elif use_sh:
    features = evaluate_sh_at(gaussians.feature, gaussians.position.detach(), indexes,
                              camera_position, indexes_sorted_unique=True)
  else:
    assert len(gaussians.feature.shape) == 2, f"Features must be (N, C) if use_sh=False, got {gaussians.feature.shape}"
    # one gather kernel, the two depth channels of render_depth assembled in front of the rows by the same call
    features = _visible_features(gaussians.feature, indexes, None, depths if render_depth else None)
    if features is not None:
      depth_in_features = render_depth
    else:
      features = gaussians.feature[indexes]

  rendering = render_projected(indexes, gaussians2d, features, depths, camera_params, config,
                               render_depth=render_depth, use_depth16=use_depth16,
                               render_median_depth=render_median_depth, mapper_front=early.get("front"),
                               before_total_sync=fill_features, features_include_depth=depth_in_features)
  return _bf16_image(rendering, gaussians.feature, use_sh, render_depth)


def _bf16_image(rendering, feature, use_sh, render_depth):
  """bf16 plain features with render_depth were rendered widened to float32 (the depth channels need it): round the
  returned image back to the features' dtype."""
  if not use_sh and render_depth and feature.dtype == torch.bfloat16:
    return replace(rendering, image=rendering.image.to(torch.bfloat16))
  return rendering


def _render_gaussians_static(gaussians, camera_params, config, use_sh, render_depth, use_depth16, render_median_depth,
                             sh_colors, overlap_capacity, overlap_total_out):
  """render_gaussians without a single host read-back (see its ``overlap_capacity``): projection with the visible
  count left on the device, the ``*_counted`` tile mapper front, the capacity-bounded back half, the rasterizer over
  the capacity-sized buffers (rows past the count are never referenced by a tile list)."""
  assert gaussians.position.dtype == torch.float32, "overlap_capacity: float32 gaussians only"
  size = camera_params.image_size
  ndc_range = (camera_params.near_plane, camera_params.far_plane)
  camera_position = camera_params.camera_position if use_sh else None
  gaussians2d, depths, indexes, count = project_to_image_static(gaussians, camera_params, config)
  front = launch_mapper_front_counted(gaussians2d.detach(), depths.detach(), count, size, config, use_depth16,
                                      ndc_range, read_back=False)
  if use_sh:
    feature, position = gaussians.feature, gaussians.position
    assert feature.is_contiguous() and position.is_contiguous() and feature.dtype == torch.float32, \
      "overlap_capacity with use_sh: contiguous float32 SH coefficients and positions"
    if sh_colors is not None:
      assert sh_colors.shape == (feature.shape[0], feature.shape[1]) and sh_colors.is_contiguous()
      pre = launch_gather_counted(sh_colors, indexes, count)
    else:
      pre = launch_sh_forward_counted(feature.detach(), position.detach(), indexes, count,
                                      camera_position.detach().to(feature.dtype).contiguous())
    features = evaluate_sh_at(feature, position.detach(), indexes, camera_position, indexes_sorted_unique=True,
                              precomputed=pre, count=count)
  else:
    assert sh_colors is None
    assert len(gaussians.feature.shape) == 2, f"Features must be (N, C) if use_sh=False, got {gaussians.feature.shape}"
    features = _visible_features(gaussians.feature, indexes, count, depths if render_depth else None)
    assert features is not None, "overlap_capacity without SH: dense contiguous float32 or bfloat16 features"
  if render_depth and use_sh:
    features = torch.cat([depths, depths ** 2, features], dim=1)
  overlap_to_point, tile_ranges = map_front_to_tiles_capped(gaussians2d, count, front, size, config, overlap_capacity,
                                                            overlap_total_out)
  ranges = tile_ranges.view(-1, 2)
  raster = rasterize_with_tiles(gaussians2d, features, tile_overlap_ranges=ranges, overlap_to_point=overlap_to_point,
                                image_size=size, config=config)
  image, depth_image, depth_var = raster.image, None, None
  if render_depth:
    depth2, image = _SplitDepthChannels.apply(image)
    depth_image, depth_var = compute_depth_variance(depth2, raster.image_weight)
  return _bf16_image(Rendering(
    image=image, image_weight=raster.image_weight, depth=depth_image, depth_var=depth_var,
    median_depth=(_median_depth(gaussians2d, depths, overlap_to_point, ranges, camera_params, config)
                  if render_median_depth else None),
    points_in_view=indexes, point_depth=depths, gaussians2d=gaussians2d,
    point_visibility=raster.visibility if config.compute_visibility else None,
    point_heuristic=raster.point_heuristic if config.compute_point_heuristic else None,
    camera=camera_params, config=config, points_in_view_count=count), gaussians.feature, use_sh, render_depth)


class _VisibleFeatures(torch.autograd.Function):
  """The plain (non-SH) feature rows of the visible set, optionally behind the two depth channels of render_depth:
  ``[depth, depth^2, feature[indexes]]`` assembled by ONE gather kernel (gs_gather_rows_strided) instead of
  ``feature[indexes]`` + ``torch.cat`` (renderer.py:152-153, 199-200 of the reference), the backward ONE scatter
  (gs_scatter_rows_strided: the indexes are unique, no atomics, no sort) instead of index_put with accumulate + the
  slices of the cat.  bfloat16 rows (no depth channels) go through the 2-byte entry points *_u16.  ``count`` (optional, (1,) int32 on the device): only the first count[0] rows of ``indexes`` are
  valid (read-back free path); rows past it are left uninitialised / ignored."""

  @staticmethod
  def forward(ctx, feature, indexes, count, depths):
    import ctypes
    from . import _native as N
    v, c = indexes.shape[0], feature.shape[1]
    extra = 0 if depths is None else 2
    out = torch.empty((v, c + extra), dtype=feature.dtype, device=feature.device)
    u16 = feature.dtype == torch.bfloat16
    N.call("gs_gather_rows_strided_u16" if u16 else "gs_gather_rows_strided", ctypes.c_int64(v), ctypes.c_int32(c), N.ptr(feature), N.ptr(indexes),
           N.ptr(count), N.ptr(out), ctypes.c_int32(c + extra), ctypes.c_int32(extra), N.stream_ptr(feature.device))
    if depths is not None:
      out[:, 0:1] = depths
      out[:, 1:2] = depths * depths
    ctx.rows, ctx.extra = feature.shape[0], extra
    ctx.save_for_backward(indexes, count, depths)
    return out

  @staticmethod
  def backward(ctx, g):
    import ctypes
    from . import _native as N
    indexes, count, depths = ctx.saved_tensors
    g = g.contiguous()
    v, width = g.shape
    c = width - ctx.extra
    g_feature = g_depths = None
    if ctx.needs_input_grad[0]:
      g_feature = torch.empty((ctx.rows, c), dtype=g.dtype, device=g.device)
      N.call("gs_scatter_rows_strided_u16" if g.dtype == torch.bfloat16 else "gs_scatter_rows_strided", ctypes.c_int64(v), ctypes.c_int32(c), N.ptr(g), ctypes.c_int32(width),
             ctypes.c_int32(ctx.extra), N.ptr(indexes), N.ptr(count), ctypes.c_int64(ctx.rows), N.ptr(g_feature),
             N.stream_ptr(g.device))
    if depths is not None and ctx.needs_input_grad[3]:
      g_depths = g[:, 0:1] + 2.0 * depths * g[:, 1:2]
    return g_feature, None, None, g_depths


def _visible_features(feature, indexes, count=None, depths=None):
  """feature[indexes] (with the depth channels in front when ``depths`` is given) through the kernels above when the
  features are dense contiguous float32 or bfloat16 on the GPU; None otherwise (the caller indexes with torch).
  bfloat16 with ``depths``: the gathered rows widened to float32 behind the f32 depth channels."""
  if not (feature.is_cuda and feature.ndim == 2 and feature.is_contiguous()):
    return None
  if feature.dtype == torch.bfloat16 and (depths is None or depths.dtype == torch.float32):
    rows = _VisibleFeatures.apply(feature, indexes.contiguous(), count, None)
    return rows if depths is None else torch.cat([depths, depths * depths, rows.float()], dim=1)
  if feature.dtype == torch.float32 and (depths is None or depths.dtype == torch.float32):
    return _VisibleFeatures.apply(feature, indexes.contiguous(), count, depths)
  return None


class _SplitDepthChannels(torch.autograd.Function):
  """(H, W, 2 + C) blended [depth, depth^2, features] -> contiguous (H, W, 2) and (H, W, C).

  The reference slices (renderer.py:215-222): two strided views of one tensor, every later elementwise operation of the
  caller (a loss over a 34-channel 4K image, say) then runs on a strided view, and autograd's backward of the two slices
  is two zero-filled full-size tensors plus their sum — at config 4 that glue cost 7 ms of a 16.6 ms frame.  Here the two
  parts are copied out once (same values) and the backward writes both gradients into ONE uninitialised full-size
  tensor: each element exactly once, no zero fill, no add."""

  @staticmethod
  def forward(ctx, image):
    ctx.shape, ctx.opts = image.shape, dict(dtype=image.dtype, device=image.device)
    ctx.native = image.is_cuda and image.dtype == torch.float32 and image.is_contiguous()
    if not ctx.native:
      return image[..., :2].contiguous(), image[..., 2:].contiguous()
    import ctypes
    from . import _native as N
    h, w, f = image.shape
    depth2 = torch.empty((h, w, 2), **ctx.opts)
    rest = torch.empty((h, w, f - 2), **ctx.opts)
    N.call("gs_split_channels", ctypes.c_int64(h * w), ctypes.c_int32(f), ctypes.c_int32(2), N.ptr(image), N.ptr(depth2),
           N.ptr(rest), N.stream_ptr(image.device))
    return depth2, rest

  @staticmethod
  def backward(ctx, g_depth, g_feat):
    g = torch.empty(ctx.shape, **ctx.opts)
    if ctx.native:
      import ctypes
      from . import _native as N
      h, w, f = ctx.shape
      N.call("gs_merge_channels", ctypes.c_int64(h * w), ctypes.c_int32(f), ctypes.c_int32(2),
             N.ptr(None if g_depth is None else g_depth.contiguous()),
             N.ptr(None if g_feat is None else g_feat.contiguous()), N.ptr(g), N.stream_ptr(g.device))
      return g
    if g_depth is None:
      g[..., :2].zero_()
    else:
      g[..., :2].copy_(g_depth)
    if g_feat is None:
      g[..., 2:].zero_()
    else:
      g[..., 2:].copy_(g_feat)
    return g


def compute_depth_variance(depth_depthsq, weight, eps=1e-6):
  """(H, W, 2) blended [depth, depth^2] and (H, W) weight -> weight-normalised depth and its variance
  (renderer.py:173-180 of the reference)."""
  norm = weight + eps
  mean = depth_depthsq[..., 0] / norm
  return mean, depth_depthsq[..., 1] / norm - mean ** 2


def _median_depth(gaussians2d, depths, overlap_to_point, ranges, camera_params, config):
  """Depth of the first gaussian at which the accumulated alpha reaches one half: the quantile mode of the
  rasterizer (no blending, saturate_threshold 0.5).  Differentiable w.r.t. the point depths (each pixel's gradient
  goes to the depth of the gaussian it selected; the selection itself is piecewise constant, so the packed 2D
  gaussians get no gradient and are detached) — the reference's quantile mode is forward only (SURVEY Q7, 8f rank 3)."""
  quantile = replace(config, use_alpha_blending=False, saturate_threshold=0.5,
                     compute_visibility=False, compute_point_heuristic=False, differentiable_weight=False)
  raster = rasterize_with_tiles(gaussians2d.detach(), depths, tile_overlap_ranges=ranges,
                                overlap_to_point=overlap_to_point, image_size=camera_params.image_size,
                                config=quantile)
  return raster.image.squeeze(-1)


def render_projected(indexes: torch.Tensor, gaussians2d: torch.Tensor,
                     features: torch.Tensor, depths: torch.Tensor,
                     camera_params: CameraParams, config: RasterConfig,
                     render_depth: bool = False, use_depth16: bool = False,
                     render_median_depth: bool = False, use_ndc_depth: bool = False,
                     mapper_front=None, before_total_sync=None, features_include_depth: bool = False):
  """Tile-map and rasterize gaussians that are already projected (renderer.py:183-231 of the reference).
  Gaussians are ordered by NDC depth inside every tile; depth features stay linear unless use_ndc_depth.
  ``mapper_front`` (extension): the front half of the tile mapping of exactly these gaussians when render_gaussians has
  already enqueued it (mapper.tile_mapper.launch_mapper_front_counted); ``before_total_sync``: see _map_to_tiles (called exactly
  once before the rasterizer is enqueued); ``features_include_depth``: the caller has already put the two depth channels
  in front of the feature rows (render_gaussians' plain-feature path assembles them with its gather kernel)."""
  size = camera_params.image_size
  ndc_range = (camera_params.near_plane, camera_params.far_plane)

  if render_depth and not features_include_depth:   # two extra leading channels: depth and depth^2, blended like any other feature
    if before_total_sync is not None:   # the features are read right here: their kernel cannot wait for the mapper
      before_total_sync()
      before_total_sync = None
    if use_ndc_depth:
      depths = ndc_depth(depths, *ndc_range)
    features = torch.cat([depths, depths ** 2, features], dim=1)

  # gaussians are ordered by NDC depth inside every tile; the key kernel forms it from the linear depth
  if render_depth and use_ndc_depth:
    if before_total_sync is not None:
      before_total_sync()
    overlap_to_point, tile_ranges = map_to_tiles(gaussians2d, depths, image_size=size, config=config,
                                                 use_depth16=use_depth16)
  else:
    overlap_to_point, tile_ranges = _map_to_tiles(gaussians2d, depths, size, config, use_depth16, ndc_range=ndc_range,
                                                  front=mapper_front, before_total_sync=before_total_sync)
  ranges = tile_ranges.view(-1, 2)
  raster = rasterize_with_tiles(gaussians2d, features, tile_overlap_ranges=ranges,
                                overlap_to_point=overlap_to_point, image_size=size, config=config)

  image, depth_image, depth_var = raster.image, None, None
  if render_depth:
    depth2, image = _SplitDepthChannels.apply(image)
    depth_image, depth_var = compute_depth_variance(depth2, raster.image_weight)

  return Rendering(
    image=image, image_weight=raster.image_weight, depth=depth_image, depth_var=depth_var,
    median_depth=(_median_depth(gaussians2d, depths, overlap_to_point, ranges, camera_params, config)
                  if render_median_depth else None),
    points_in_view=indexes, point_depth=depths, gaussians2d=gaussians2d,
    point_visibility=raster.visibility if config.compute_visibility else None,
    point_heuristic=raster.point_heuristic if config.compute_point_heuristic else None,
    camera=camera_params, config=config)


def viewspace_gradient(gaussians2d: torch.Tensor):
  assert gaussians2d.shape[1] == 7, f"Expected packed 2D gaussians (N, 7), got {gaussians2d.shape}"
  assert gaussians2d.grad is not None, \
    "Expected gradients on gaussians2d, run backward first with gaussians2d.retain_grad()"
  xy_grad = gaussians2d.grad[:, :2]
  return torch.norm(xy_grad, dim=1)
