"""Configuration and parameter containers of the render path.

Mirrors taichi_splatting/data_types.py (RasterConfig :10-39, Gaussians3D :52-94,
Gaussians2D :100-121) field for field.  The reference builds the two containers with
``tensordict.tensorclass``; tensordict is not a dependency here, so the handful of
tensorclass behaviours its callers rely on (``batch_size=``, ``.to``, ``.cuda``,
``.requires_grad_``, index/mask ``__getitem__``, ``.apply``, ``dataclasses.replace``,
``to_tensordict``/``from_tensordict``) are provided by a small dataclass mixin.
"""
from dataclasses import dataclass, fields, replace
from typing import Any, Callable, Dict, Optional

import torch
from beartype import beartype
from beartype.typing import Tuple


@beartype
@dataclass(frozen=True, eq=True, kw_only=True)
class RasterConfig:
  tile_size: int = 16

  # pixels per thread in the reference's backward kernel; accepted and validated for
  # compatibility, the sm_100a kernels choose their own pixel ownership (results are
  # independent of it, see DESIGN.md)
  pixel_stride: Tuple[int, int] = (2, 2)

  # clamp position to within this margin of the image for the affine jacobian
  clamp_margin: float = 0.15

  # antialiased (box-integrated logistic approximation) gaussian evaluation
  antialias: bool = False

  # blur added to the projected covariance diagonal
  blur_cov: float = 0.3

  clamp_max_alpha: float = 0.99
  alpha_threshold: float = 1. / 255.

  # backward pass stops accumulating once a pixel's weight passes this
  saturate_threshold: float = 0.9999

  # False: pick the feature of the first gaussian at which the accumulated weight
  # reaches 1 - saturate_threshold (quantile / median rendering, forward only)
  use_alpha_blending: bool = True

  compute_point_heuristic: bool = False  # split / prune statistics (backward)
  compute_visibility: bool = False       # per gaussian sum of blend weights (forward)

  # (extension) image_weight is a differentiable output: its gradient reaches the gaussians and the heuristics as
  # that of one more feature channel of ones would (background compositing, mask losses, depth / (W + eps)).  Off
  # by default because it changes the gradient of code that already uses image_weight.  Alpha blending only: in
  # quantile mode image_weight is W > 0 and stays non-differentiable.
  differentiable_weight: bool = False


def check_packed3d(packed_gaussians: torch.Tensor):
  assert len(packed_gaussians.shape) == 2 and packed_gaussians.shape[1] == 11, \
    f"Expected shape (N, 11), got {packed_gaussians.shape}"


def check_packed2d(packed_gaussians: torch.Tensor):
  assert len(packed_gaussians.shape) == 2 and packed_gaussians.shape[1] == 7, \
    f"Expected shape (N, 7), got {packed_gaussians.shape}"


class _TensorFields:
  """The subset of tensorclass behaviour the reference's callers use."""

  def _tensor_items(self):
    return [(f.name, getattr(self, f.name)) for f in fields(self) if f.name != 'batch_size']

  def items(self):
    return self._tensor_items()

  def keys(self):
    return [k for k, _ in self._tensor_items()]

  def _check_batch(self):
    n = None
    for name, t in self._tensor_items():
      assert isinstance(t, torch.Tensor), f"{name}: expected a tensor, got {type(t)}"
      n = t.shape[0] if n is None else n
      assert t.shape[0] == n, f"{name}: leading dimension {t.shape[0]} != {n}"
    if self.batch_size is None:
      object.__setattr__(self, 'batch_size', (n,))
    else:
      bs = tuple(int(x) for x in self.batch_size)
      assert bs == (n,), f"batch_size {bs} does not match tensors of length {n}"
      object.__setattr__(self, 'batch_size', bs)

  def apply(self, fn: Callable[[torch.Tensor], torch.Tensor], batch_size=None):
    out = {k: fn(t) for k, t in self._tensor_items()}
    return type(self)(**out, batch_size=None if batch_size is None else tuple(batch_size))

  def to(self, device=None, dtype=None):
    def f(t):
      if dtype is not None and not t.is_floating_point():
        return t.to(device=device)
      return t.to(device=device, dtype=dtype)
    return self.apply(f, batch_size=self.batch_size)

  def cuda(self, device=None):
    return self.apply(lambda t: t.cuda(device), batch_size=self.batch_size)

  def cpu(self):
    return self.apply(lambda t: t.cpu(), batch_size=self.batch_size)

  def detach(self):
    return self.apply(lambda t: t.detach(), batch_size=self.batch_size)

  def clone(self):
    return self.apply(lambda t: t.clone(), batch_size=self.batch_size)

  def contiguous(self):
    return self.apply(lambda t: t.contiguous(), batch_size=self.batch_size)

  def requires_grad_(self, requires_grad: bool = True):
    for _, t in self._tensor_items():
      if t.is_floating_point():
        t.requires_grad_(requires_grad)
    return self

  @property
  def device(self):
    return self._tensor_items()[0][1].device

  @property
  def dtype(self):
    return self._tensor_items()[0][1].dtype

  @property
  def shape(self):
    return torch.Size(self.batch_size)

  def __len__(self):
    return self.batch_size[0]

  def __getitem__(self, index):
    return self.apply(lambda t: t[index], batch_size=None)

  def to_tensordict(self):
    from .tensor_dict import TensorDict
    return TensorDict(dict(self._tensor_items()), batch_size=self.batch_size)

  def to_dict(self) -> Dict[str, torch.Tensor]:
    return dict(self._tensor_items())

  @classmethod
  def from_tensordict(cls, tensors):
    names = [f.name for f in fields(cls) if f.name != 'batch_size']
    return cls(**{k: tensors[k] for k in names})

  from_dict = from_tensordict


@dataclass
class Gaussians3D(_TensorFields):
  position: torch.Tensor      # 3  - xyz
  log_scaling: torch.Tensor   # 3  - scale = exp(log_scaling)
  rotation: torch.Tensor      # 4  - quaternion, component order x y z w (taichi_lib/generic.py:418-427)
  alpha_logit: torch.Tensor   # 1  - alpha = sigmoid(alpha_logit)
  feature: torch.Tensor       # (N, C) features or (N, C, (deg+1)^2) spherical harmonics
  batch_size: Optional[Any] = None

  def __post_init__(self):
    assert self.position.shape[1] == 3, f"Expected shape (N, 3), got {self.position.shape}"
    assert self.log_scaling.shape[1] == 3, f"Expected shape (N, 3), got {self.log_scaling.shape}"
    assert self.rotation.shape[1] == 4, f"Expected shape (N, 4), got {self.rotation.shape}"
    assert self.alpha_logit.shape[1] == 1, f"Expected shape (N, 1), got {self.alpha_logit.shape}"
    self._check_batch()

  def packed(self):
    return torch.cat([self.position, self.log_scaling, self.rotation, self.alpha_logit], dim=-1)

  def shape_tensors(self):
    return (self.position, self.log_scaling, self.rotation, self.alpha_logit)

  @property
  def scale(self):
    return torch.exp(self.log_scaling)

  @property
  def alpha(self):
    return torch.sigmoid(self.alpha_logit)

  def replace(self, **kwargs):
    kwargs.setdefault('batch_size', None)
    return replace(self, **kwargs)

  def concat(self, other):
    return Gaussians3D(
      position=torch.cat([self.position, other.position], dim=0),
      log_scaling=torch.cat([self.log_scaling, other.log_scaling], dim=0),
      rotation=torch.cat([self.rotation, other.rotation], dim=0),
      alpha_logit=torch.cat([self.alpha_logit, other.alpha_logit], dim=0),
      feature=torch.cat([self.feature, other.feature], dim=0),
      batch_size=(self.batch_size[0] + other.batch_size[0],))


def inverse_sigmoid(x: torch.Tensor):
  return torch.log(x / (1 - x))


@dataclass
class Gaussians2D(_TensorFields):
  position: torch.Tensor      # 2  - xy
  z_depth: torch.Tensor       # 1  - for sorting
  log_scaling: torch.Tensor   # 2
  rotation: torch.Tensor      # 2  - unit length complex number
  alpha_logit: torch.Tensor   # (N,) - alpha = sigmoid(alpha_logit)
  feature: torch.Tensor       # (N, C) - rgb, labels, ...
  batch_size: Optional[Any] = None

  def __post_init__(self):
    self._check_batch()

  @property
  def opacity(self):
    return self.alpha_logit.sigmoid()

  @property
  def scaling(self):
    return torch.exp(self.log_scaling)

  def set_scaling(self, scaling) -> 'Gaussians2D':
    return replace(self, log_scaling=torch.log(scaling))
