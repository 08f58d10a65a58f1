"""View dependent colour from real spherical harmonics (degree 0..3).

Operator surface of taichi_splatting/spherical_harmonics.py:167-178 (``evaluate_sh_at``); the
forward / backward kernels are csrc/point_kernels.cu (replacing evaluate_sh_at_kernel and its
Taichi autodiff, :118-134 and :154-161).  Layout is channel major: (M, K, (degree+1)^2).
"""
import ctypes
import math
from typing import Optional

import torch
from beartype import beartype

from . import _native as N
from .grad_sinks import deferred_sh, grad_sink, register_grad_sink, unregister_grad_sink  # noqa: F401  (re-exported)
from .grad_sinks import flush_sh_views


def check_sh_degree(sh_features):
  assert len(sh_features.shape) == 3, f"SH features must have 3 dimensions, got {sh_features.shape}"
  n_sh = sh_features.shape[2]
  n = int(math.isqrt(n_sh))
  assert n * n == n_sh, f"SH feature count must be square, got {n_sh} ({sh_features.shape})"
  assert 0 <= n - 1 <= 3, f"SH degree must be between 0 and 3, got {n - 1}"
  return n - 1


def sh_fast_path(sh_params: torch.Tensor) -> bool:
  """Whether the batched forward (evaluate_sh_views), the counted forward / backward (render_gaussians(...,
  overlap_capacity=)), the dense backward and the deferred gradient of GradientBucket.fused_accumulation() serve these
  coefficients: float32, 3 channels, degree 0..3, i.e. (N, 3, 1 | 4 | 9 | 16).  Other shapes take the generic kernels
  (or are refused where there is no generic path)."""
  return sh_params.dtype == torch.float32 and sh_params.ndim == 3 and sh_params.shape[1] == 3 \
    and sh_params.shape[2] in (1, 4, 9, 16)


class _SHFunction(torch.autograd.Function):

  @staticmethod
  def forward(ctx, params, points, indexes, camera_pos, sorted_unique=False, precomputed=None, count=None):
    m, k, d = params.shape
    v = indexes.shape[0]
    p = N.GsSHParams(N.dtype_code(params.dtype), k, d, int(bool(sorted_unique)), m, v, 0, 0)
    ctx.count = count   # (1,) int32 on the device: only the first count[0] rows of indexes / out are valid
    if count is not None:
      assert precomputed is not None and sorted_unique and sh_fast_path(params), \
        "counted SH evaluation: precomputed f32 colours of the ascending visible set, 3 channels, degree 0..3"
    if precomputed is not None:     # evaluated ahead of time on the capacity buffers (launch_sh_forward_counted)
      assert precomputed.shape == (v, k)
      out = precomputed
    else:
      out = torch.empty((v, k), dtype=params.dtype, device=params.device)
      N.call("gs_sh_fwd", ctypes.byref(p), N.ptr(params), N.ptr(points), N.ptr(indexes), N.ptr(camera_pos),
             N.ptr(out), N.stream_ptr(params.device))
    ctx.p = p
    ctx.sorted_unique = bool(sorted_unique)
    ctx.mark_non_differentiable(indexes)
    ctx.save_for_backward(params, points, indexes, camera_pos, out)
    return out

  @staticmethod
  def backward(ctx, doutput):
    params, points, indexes, camera_pos, out = ctx.saved_tensors
    need = ctx.needs_input_grad
    dense = ctx.sorted_unique and sh_fast_path(params) and indexes.shape[0] > 0
    sink = grad_sink(params) if (need[0] and dense) else None
    g_points = torch.empty_like(points) if need[1] else None
    g_cam = torch.empty_like(camera_pos) if need[3] else None
    if sink is not None or ctx.count is not None:
      # the masked colour gradient is staged (the stage kernel reads only the forward output) and turned into
      # coefficient rows by a flush: the batch's deferred one, a one-view flush added to the sink, or (counted path
      # without a sink: render_gaussians(..., overlap_capacity=)) a one-view flush into a fresh dense gradient
      if ctx.count is not None:
        assert need[0] and not need[1] and not need[3], "counted SH backward: coefficient gradient only"
      deferred = deferred_sh(params) if sink is not None else None
      staged = deferred.staging_buffer() if deferred is not None else None
      if staged is None:
        staged = torch.empty((params.shape[0], params.shape[1]), dtype=params.dtype, device=params.device)
      p = N.GsSHParams(ctx.p.dtype, ctx.p.num_channels, ctx.p.num_coeffs, 1, ctx.p.num_points, ctx.p.num_indexes, 1, 1)
      if ctx.count is not None:
        N.call("gs_sh_bwd_stage_counted", ctypes.byref(p), N.ptr(out), N.ptr(indexes), N.ptr(doutput.contiguous()),
               N.ptr(ctx.count), N.ptr(staged), N.stream_ptr(params.device))
      else:
        N.call("gs_sh_bwd_stage", ctypes.byref(p), N.ptr(out), N.ptr(indexes), N.ptr(doutput.contiguous()),
               N.ptr(staged), N.stream_ptr(params.device))
      cam = camera_pos.detach().contiguous()
      g_params = None
      if deferred is not None:
        deferred.add(staged, cam, points.detach())
      elif sink is not None:
        flush_sh_views(sink, points.detach(), [staged], [cam], overwrite=False)
      else:
        g_params = torch.empty_like(params)
        flush_sh_views(g_params, points.detach(), [staged], [cam], overwrite=True)
      if g_points is not None or g_cam is not None:
        # position / camera gradient (eager path only): the generic kernel, no coefficient rows
        N.call("gs_sh_bwd", ctypes.byref(ctx.p), N.ptr(params), N.ptr(points), N.ptr(indexes), N.ptr(camera_pos),
               N.ptr(doutput.contiguous()), N.ptr(None), N.ptr(g_points), N.ptr(g_cam), N.stream_ptr(params.device))
      return g_params, g_points, None, g_cam, None, None, None
    g_params = torch.empty_like(params) if need[0] else None
    # only the coefficient gradient is wanted (render_gaussians detaches the positions): the kernel then takes the clamp
    # mask from the forward output and never reads the coefficient rows
    from_out = int(dense and need[0] and not need[1] and not need[3])
    coeffs = out if from_out else params
    p = N.GsSHParams(ctx.p.dtype, ctx.p.num_channels, ctx.p.num_coeffs, ctx.p.indexes_sorted_unique, ctx.p.num_points,
                     ctx.p.num_indexes, 0, from_out)
    N.call("gs_sh_bwd", ctypes.byref(p), N.ptr(coeffs), N.ptr(points), N.ptr(indexes),
                              N.ptr(camera_pos), N.ptr(doutput.contiguous()), N.ptr(g_params), N.ptr(g_points),
                              N.ptr(g_cam), N.stream_ptr(params.device))
    return g_params, g_points, None, g_cam, None, None, None


def launch_sh_forward_counted(sh_params, positions, indexes_capacity, count_device, camera_pos) -> torch.Tensor:
  """Enqueue the SH evaluation for a visible set whose SIZE is still on the device: ``indexes_capacity`` (N,) holds
  the valid indexes in its first ``count_device[0]`` rows.  Returns the (N, K) output buffer; rows past the count are
  uninitialised.  Used by render_gaussians to keep the GPU busy across the host read-back of the visible count."""
  check_sh_degree(sh_params)
  m, k, d = sh_params.shape
  cap = indexes_capacity.shape[0]
  p = N.GsSHParams(N.dtype_code(sh_params.dtype), k, d, 1, m, cap, 0, 0)
  out = torch.empty((cap, k), dtype=sh_params.dtype, device=sh_params.device)
  N.call("gs_sh_fwd_counted", ctypes.byref(p), N.ptr(sh_params), N.ptr(positions), N.ptr(indexes_capacity),
         N.ptr(camera_pos), N.ptr(count_device), N.ptr(out), N.stream_ptr(sh_params.device))
  return out


def evaluate_sh_views(sh_params: torch.Tensor, positions: torch.Tensor, camera_positions) -> list:
  """Colours of ALL gaussians for every view of a batch, one dense (M, K) tensor per camera position (extension, not
  in the reference): the coefficient rows are read once per batch instead of once per view (gs_sh_fwd_views; f32,
  K = 3, degree 0..3).  Pass a view's tensor to ``render_gaussians(..., sh_colors=...)``, which gathers the visible
  rows and builds the same autograd node as ``evaluate_sh_at`` (gradients reach ``sh_params``).  Worth it when most
  gaussians are in view in most views; values are those of ``evaluate_sh_at``."""
  check_sh_degree(sh_params)
  N.require_cuda(sh_params, positions)
  m, k, d = sh_params.shape
  assert sh_fast_path(sh_params), \
    f"evaluate_sh_views: float32, 3 channels, degree 0..3 (got {sh_params.dtype}, {tuple(sh_params.shape)})"
  params = sh_params.detach().contiguous()
  pos = positions.detach().to(torch.float32).contiguous()
  cams = [c.detach().to(torch.float32).contiguous() for c in camera_positions]
  outs = [torch.empty((m, k), dtype=torch.float32, device=sh_params.device) for _ in cams]
  p = N.GsSHParams(N.GS_F32, k, d, 1, m, 0, 0, 0)
  for s in range(0, len(cams), 16):
    nv = len(cams[s:s + 16])
    arr = ctypes.c_void_p * nv
    N.call("gs_sh_fwd_views", ctypes.byref(p), ctypes.c_int32(nv), N.ptr(params), N.ptr(pos),
           arr(*[c.data_ptr() for c in cams[s:s + 16]]), arr(*[o.data_ptr() for o in outs[s:s + 16]]),
           N.stream_ptr(sh_params.device))
  return outs


def launch_sh_forward_into(sh_params, positions, indexes, camera_pos, out):
  """Enqueue the SH evaluation of ``indexes`` into the existing (V, K) buffer ``out`` (no autograd node: pair it with
  ``evaluate_sh_at(..., precomputed=out)``; the node may be built before this launch, the data is only read by kernels
  enqueued later on the same stream)."""
  m, k, d = sh_params.shape
  p = N.GsSHParams(N.dtype_code(sh_params.dtype), k, d, 1, m, indexes.shape[0], 0, 0)
  N.call("gs_sh_fwd", ctypes.byref(p), N.ptr(sh_params), N.ptr(positions), N.ptr(indexes), N.ptr(camera_pos),
         N.ptr(out), N.stream_ptr(sh_params.device))


def launch_gather_into(dense: torch.Tensor, indexes: torch.Tensor, out: torch.Tensor):
  """``out[:] = dense[indexes]`` (rows of 3 floats), enqueued; see launch_sh_forward_into."""
  N.call("gs_gather_rows_counted", ctypes.c_int64(indexes.shape[0]), ctypes.c_int32(dense.shape[1]), N.ptr(dense),
         N.ptr(indexes), N.ptr(None), N.ptr(out), N.stream_ptr(dense.device))


def launch_gather_counted(dense: torch.Tensor, indexes_capacity: torch.Tensor, count_device: torch.Tensor) -> torch.Tensor:
  """``dense[indexes]`` for a visible set whose SIZE is still on the device (see launch_sh_forward_counted): returns
  the (capacity, K) buffer, rows past the count uninitialised."""
  cap, k = indexes_capacity.shape[0], dense.shape[1]
  out = torch.empty((cap, k), dtype=dense.dtype, device=dense.device)
  N.call("gs_gather_rows_counted", ctypes.c_int64(cap), ctypes.c_int32(k), N.ptr(dense), N.ptr(indexes_capacity),
         N.ptr(count_device), N.ptr(out), N.stream_ptr(dense.device))
  return out


@beartype
def evaluate_sh_at(sh_params: torch.Tensor,   # M, K, (degree + 1)^2  (usually K=3, for RGB)
                   positions: torch.Tensor,   # M, 3
                   indexes: torch.Tensor,     # V   (int64 indexes into the M gaussians)
                   camera_pos: torch.Tensor,  # 3
                   indexes_sorted_unique: bool = False,
                   precomputed: Optional[torch.Tensor] = None,
                   count: Optional[torch.Tensor] = None
                   ) -> torch.Tensor:         # V, K
  """``indexes_sorted_unique`` (extension, not in the reference signature): promise that ``indexes`` is strictly
  ascending, as the visible set returned by project_to_image is; the backward then writes dense gradient rows
  without atomics or a memset (csrc/point_kernels.cu sh_bwd_dense_kernel).  Results are identical.
  ``precomputed``: the forward values already evaluated by launch_sh_forward_counted for exactly these inputs; the
  call then only builds the autograd node.  ``count`` (with ``precomputed``): a (1,) int32 CUDA tensor — ``indexes`` and
  ``precomputed`` are capacity-sized and only their first ``count[0]`` rows are valid (project_to_image_static); the
  backward then reads the count on the device as well."""
  check_sh_degree(sh_params)
  N.require_cuda(sh_params, positions, indexes, camera_pos)
  dtype = sh_params.dtype
  return _SHFunction.apply(sh_params.contiguous(), positions.to(dtype).contiguous(),
                           indexes.to(torch.int64).contiguous(), camera_pos.to(dtype).contiguous(),
                           indexes_sorted_unique, precomputed, count)
