"""``Rendering``: what ``render_gaussians`` returns.

Field and property names are the reference's (taichi_splatting/renderer.py:27-131) because callers — the
external trainer and viewer — read them; the implementation is organised around three small helpers
(``_to_ndc``, ``_stat_column``, ``_require``) instead of one property body per quantity.
"""
import dataclasses
from functools import cached_property
from numbers import Integral

import torch
from beartype.typing import Optional, Tuple

from .data_types import RasterConfig
from .perspective import CameraParams
from .torch_lib.projection import ndc_depth as _ndc

_NO_STATS = "No point heuristic information available (use config.compute_point_heuristic=True)"
_NO_VISIBILITY = "No visibility information available (use config.compute_visibility=True)"


@dataclasses.dataclass(frozen=True, kw_only=True)
class Rendering:
  """Images plus the per point by-products of one rendered view.

  Shapes: H, W image size; C feature channels; V gaussians inside the view frustum.
  ``depth`` / ``depth_var`` exist only for ``render_depth=True``, ``median_depth`` only for
  ``render_median_depth=True``.  ``point_heuristic`` is allocated by the forward pass and FILLED BY THE BACKWARD
  pass (rasterizer/function.py:52,89 of the reference), so read it after ``loss.backward()``.
  """
  # pixel space
  image: torch.Tensor                              # (H, W, C)
  image_weight: torch.Tensor                       # (H, W) accumulated alpha (differentiable with RasterConfig.differentiable_weight)
  depth: Optional[torch.Tensor] = None             # (H, W)
  depth_var: Optional[torch.Tensor] = None         # (H, W)
  median_depth: Optional[torch.Tensor] = None      # (H, W)

  # point space (rows follow points_in_view)
  points_in_view: torch.Tensor                     # (V,) int64 indexes into the input gaussians, ascending
  point_depth: torch.Tensor                        # (V, 1) camera space depth
  gaussians2d: torch.Tensor                        # (V, 7) mean, axis, sigma, alpha
  point_visibility: Optional[torch.Tensor] = None  # (V,) summed blend weight
  point_heuristic: Optional[torch.Tensor] = None   # (V, 2) prune cost, split score
  # (extension) render_gaussians(..., overlap_capacity=): the point space tensors keep N rows, the first
  # points_in_view_count[0] of them valid — V stays on the device ((1,) int32) so that nothing synchronises
  points_in_view_count: Optional[torch.Tensor] = None

  camera: CameraParams
  config: RasterConfig

  # ------------------------------------------------------------------ helpers
  def _to_ndc(self, linear_depth: torch.Tensor) -> torch.Tensor:
    return _ndc(linear_depth, self.camera.near_plane, self.camera.far_plane)

  def _require(self, value, message):
    assert value is not None, message
    return value

  def _stat_column(self, column: int) -> torch.Tensor:
    assert self.config.compute_point_heuristic, _NO_STATS
    return self.point_heuristic[:, column]

  # ------------------------------------------------------------------ depth in normalised device coordinates
  @cached_property
  def ndc_depth(self) -> torch.Tensor:
    return self._to_ndc(self.depth)

  @cached_property
  def ndc_median_depth(self) -> torch.Tensor:
    return self._to_ndc(self.median_depth)

  @property
  def ndc_point_depth(self) -> torch.Tensor:
    return self._to_ndc(self.point_depth)

  # ------------------------------------------------------------------ per point geometry in the image
  @property
  def point_scale(self) -> torch.Tensor:
    return self.gaussians2d[:, 4:6]        # sigma along the major / minor axis, pixels

  @property
  def point_opacity(self) -> torch.Tensor:
    return self.gaussians2d[:, 6]

  @property
  def point_radii(self) -> torch.Tensor:
    return self.point_scale.amax(dim=1)

  @property
  def gaussian_scale(self) -> torch.Tensor:
    """How many sigmas the culling ellipse extends: the level set alpha * pdf = alpha_threshold
    (3DGS uses a constant 3)."""
    return (2 * (self.point_opacity / self.config.alpha_threshold).log()).sqrt()

  # ------------------------------------------------------------------ densification statistics (after backward)
  @property
  def prune_cost(self) -> torch.Tensor:
    return self._stat_column(0)

  @property
  def split_score(self) -> torch.Tensor:
    return self._stat_column(1)

  # ------------------------------------------------------------------ visibility
  @cached_property
  def visible_mask(self) -> torch.Tensor:
    """(V,) bool: the point contributed blend weight to at least one pixel."""
    return self._require(self.point_visibility, _NO_VISIBILITY) > 0

  @cached_property
  def visible_indices(self) -> torch.Tensor:
    return self.points_in_view[self.visible_mask]

  @cached_property
  def visible(self) -> Tuple[torch.Tensor, torch.Tensor]:
    """(indexes into the input gaussians, their visibility) for the visible points only."""
    return self.visible_indices, self._require(self.point_visibility, _NO_VISIBILITY)[self.visible_mask]

  # ------------------------------------------------------------------ misc
  @property
  def image_size(self) -> Tuple[Integral, Integral]:
    return self.camera.image_size

  @property
  def num_points(self) -> int:
    return self.points_in_view.shape[0]

  def detach(self) -> "Rendering":
    """Copy with every tensor (and the camera) cut from the autograd graph."""
    values = {f.name: getattr(self, f.name) for f in dataclasses.fields(self)}
    return Rendering(**{k: (v.detach() if hasattr(v, "detach") else v) for k, v in values.items()})
