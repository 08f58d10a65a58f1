"""ctypes binding of libgsplat_b200.so (include/gsplat_b200.h).

There is no CPU or eager-torch fallback behind these functions: if the library has not been built
(``python -m taichi_gaussian_rasterizer_b200.csrc.build`` / ``__graft_entry__.build()``) or a
tensor is not a CUDA tensor, the call raises.  torch is used for device memory and streams only.
"""
import ctypes
from pathlib import Path

import torch

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libgsplat_b200.so"

GS_F32, GS_F64, GS_BF16 = 0, 1, 2

EXPORTS = [
  "gs_abi_version", "gs_last_error_string",
  "gs_project_fwd_workspace_bytes", "gs_project_fwd", "gs_project_bwd", "gs_project_bwd_counted",
  "gs_sh_fwd", "gs_sh_fwd_counted", "gs_sh_bwd", "gs_sh_bwd_stage", "gs_sh_bwd_stage_counted", "gs_sh_bwd_flush", "gs_sh_fwd_views", "gs_gather_rows_counted", "gs_gather_rows_strided", "gs_scatter_rows_strided", "gs_gather_rows_strided_u16", "gs_scatter_rows_strided_u16", "gs_split_channels", "gs_merge_channels",
  "gs_tile_count", "gs_full_cumsum_workspace_bytes", "gs_full_cumsum", "gs_full_cumsum_counted", "gs_tile_emit_keys",
  "gs_radix_sort_pairs_workspace_bytes", "gs_radix_sort_pairs", "gs_radix_sort_pairs_counted", "gs_find_ranges",
  "gs_depth_keys", "gs_depth_keys_counted", "gs_tile_count_perm", "gs_tile_count_perm_counted", "gs_tile_emit_tiles", "gs_find_ranges_tiles",
  "gs_tile_emit_tiles_capped", "gs_tile_emit_tiles_capped_counted", "gs_find_ranges_tiles_counted",
  "gs_raster_workspace_bytes", "gs_raster_fwd", "gs_raster_bwd", "gs_raster_bwd_with_weight",
  "gs_opt_update_visibility", "gs_opt_accumulate_weight", "gs_opt_step",
  "gs_morton_codes", "gs_camera_position",
  "gs_multimem_all_reduce_flag_words", "gs_multimem_all_reduce", "gs_cross_rank_barrier",
]


class GsProjectParams(ctypes.Structure):
  _fields_ = [("dtype", ctypes.c_int32), ("image_width", ctypes.c_int32), ("image_height", ctypes.c_int32),
              ("accumulate_grads", ctypes.c_int32), ("num_points", ctypes.c_int64), ("near_plane", ctypes.c_double), ("far_plane", ctypes.c_double),
              ("blur_cov", ctypes.c_double), ("clamp_margin", ctypes.c_double),
              ("alpha_threshold", ctypes.c_double)]


class GsSHParams(ctypes.Structure):
  _fields_ = [("dtype", ctypes.c_int32), ("num_channels", ctypes.c_int32), ("num_coeffs", ctypes.c_int32),
              ("indexes_sorted_unique", ctypes.c_int32), ("num_points", ctypes.c_int64),
              ("num_indexes", ctypes.c_int64), ("accumulate_params", ctypes.c_int32), ("params_is_forward_output", ctypes.c_int32)]


class GsTileParams(ctypes.Structure):
  _fields_ = [("image_width", ctypes.c_int32), ("image_height", ctypes.c_int32), ("tile_size", ctypes.c_int32),
              ("use_depth16", ctypes.c_int32), ("num_points", ctypes.c_int64),
              ("alpha_threshold", ctypes.c_double)]


class GsRasterParams(ctypes.Structure):
  _fields_ = [("dtype", ctypes.c_int32), ("image_width", ctypes.c_int32), ("image_height", ctypes.c_int32),
              ("tile_size", ctypes.c_int32), ("num_features", ctypes.c_int32), ("antialias", ctypes.c_int32),
              ("use_alpha_blending", ctypes.c_int32), ("compute_visibility", ctypes.c_int32),
              ("compute_point_heuristic", ctypes.c_int32), ("points_requires_grad", ctypes.c_int32),
              ("features_requires_grad", ctypes.c_int32), ("emulate_stale_tail", ctypes.c_int32),
              ("pixel_stride_x", ctypes.c_int32), ("pixel_stride_y", ctypes.c_int32),
              ("workspace_holds_packed", ctypes.c_int32), ("kernel_variant", ctypes.c_int32),
              ("num_points", ctypes.c_int64), ("num_overlaps", ctypes.c_int64),
              ("clamp_max_alpha", ctypes.c_double), ("alpha_threshold", ctypes.c_double),
              ("saturate_threshold", ctypes.c_double), ("forward_exit_transmittance", ctypes.c_double)]


class GsOptParams(ctypes.Structure):
  _fields_ = [("algorithm", ctypes.c_int32), ("group_type", ctypes.c_int32), ("dims", ctypes.c_int32),
              ("bias_correction", ctypes.c_int32), ("num_points", ctypes.c_int64), ("num_visible", ctypes.c_int64),
              ("lr", ctypes.c_double), ("beta1", ctypes.c_double), ("beta2", ctypes.c_double), ("eps", ctypes.c_double),
              ("grad_scale", ctypes.c_double), ("vis_smooth", ctypes.c_double)]


_lib = None


def use_library(path):
  """Load a differently built copy of the library instead of the default one (benchmarks/fast_math_cost.py: the build
  without --use_fast_math).  Must be called before the first operator runs."""
  global LIB_PATH
  assert _lib is None, "the library is already loaded"
  LIB_PATH = Path(path)


def lib():
  global _lib
  if _lib is None:
    if not LIB_PATH.exists():
      raise RuntimeError(
        f"{LIB_PATH} is missing: the sm_100a extension has not been built. Run "
        "`python -m taichi_gaussian_rasterizer_b200.csrc.build` (or __graft_entry__.build()). "
        "There is no CPU fallback.")
    l = ctypes.CDLL(str(LIB_PATH))
    l.gs_last_error_string.restype = ctypes.c_char_p
    for name in ("gs_project_fwd_workspace_bytes", "gs_full_cumsum_workspace_bytes",
                 "gs_radix_sort_pairs_workspace_bytes", "gs_raster_workspace_bytes"):
      getattr(l, name).restype = ctypes.c_size_t
    l.gs_full_cumsum_workspace_bytes.argtypes = [ctypes.c_int64, ctypes.c_int32]
    l.gs_radix_sort_pairs_workspace_bytes.argtypes = [ctypes.c_int64, ctypes.c_int32, ctypes.c_int32,
                                                      ctypes.c_int32]
    _lib = l
  return _lib


def check(rc: int, what: str):
  if rc != 0:
    msg = lib().gs_last_error_string().decode("utf-8", "replace")
    raise RuntimeError(f"{what} failed ({rc}): {msg}")


class StageTimer:
  """Optional per-entry-point device timing: CUDA events recorded on the launching stream around each
  C-ABI call (used by bench.py for the per-kernel roofline; off by default)."""

  def __init__(self):
    self.records = []   # (name, start_event, end_event)

  def summary(self):
    """name -> (calls, total_ms); synchronises."""
    torch.cuda.synchronize()
    out = {}
    for name, a, b in self.records:
      n, t = out.get(name, (0, 0.0))
      out[name] = (n + 1, t + a.elapsed_time(b))
    return out

  def reset(self):
    self.records = []


_timer = None


def set_stage_timer(timer):
  global _timer
  _timer = timer
  return timer


class StreamHandle(ctypes.c_void_p):
  """A ``cudaStream_t`` for the C ABI that remembers which device it belongs to (see ``call``)."""
  index = None


def call(name: str, *args):
  """Invoke an entry point of the library, raising RuntimeError with its message on failure.

  Device guard: the library launches on the calling thread's CURRENT device, while the pointers and the stream belong
  to the tensors' device.  The stream handle made by ``stream_ptr(device)`` carries that device's index; when it is
  not the current device the call (and the stage timer's events) run inside ``torch.cuda.device(index)``, as torch's
  own operators do.  The common case (same device) costs one integer comparison."""
  fn = getattr(lib(), name)
  index = None
  for a in reversed(args):   # the stream is the last argument of every launching entry point
    if isinstance(a, StreamHandle):
      index = a.index
      break
  if index is not None and index != torch.cuda.current_device():
    with torch.cuda.device(index):
      rc = _invoke(fn, name, args)
  else:
    rc = _invoke(fn, name, args)
  check(rc, name)


def _invoke(fn, name, args):
  if _timer is None:
    return fn(*args)
  a = torch.cuda.Event(enable_timing=True)
  b = torch.cuda.Event(enable_timing=True)
  a.record()
  rc = fn(*args)
  b.record()
  _timer.records.append((name, a, b))
  return rc


def dtype_code(dtype: torch.dtype, raster: bool = False) -> int:
  """GsDtype of ``dtype``.  ``raster``: the feature dtype of a rasterizer call, which may also be bfloat16 (GS_BF16:
  bf16 features / image, f32 geometry and gradients); every other operator is float32 / float64 only."""
  if dtype == torch.float32:
    return GS_F32
  if dtype == torch.float64:
    return GS_F64
  if raster and dtype == torch.bfloat16:
    return GS_BF16
  raise TypeError(f"unsupported dtype {dtype}: the kernels are float32 / float64"
                  + (" (the rasterizer's features may also be bfloat16)" if raster else ""))


def require_cuda(*tensors):
  """Every operator of this package runs on the GPU only; fail loudly otherwise (no CPU fallback)."""
  for t in tensors:
    if t is not None and not t.is_cuda:
      raise RuntimeError("expected a CUDA tensor: this package runs on sm_100a only, there is no CPU path "
                         f"(got device {t.device})")


def ptr(t):
  """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
  if t is None:
    return ctypes.c_void_p(0)
  if not t.is_cuda:
    raise RuntimeError("expected a CUDA tensor: this package runs on sm_100a only, there is no CPU path "
                       f"(got device {t.device})")
  if not t.is_contiguous():
    raise RuntimeError("expected a contiguous tensor")
  return ctypes.c_void_p(t.data_ptr())


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream_ptr(device=None):
  """The current CUDA stream of ``device`` as a ``cudaStream_t`` (a StreamHandle: ``call`` reads the device index off
  it).  torch.cuda.current_stream() builds a Stream object (10 us, fourteen times per frame); the raw handle is all
  the C ABI needs."""
  if device is None:
    index = torch.cuda.current_device()
  else:
    index = device.index if isinstance(device, torch.device) else int(device)
    if index is None:
      index = torch.cuda.current_device()
  if _raw_stream is not None:
    h = StreamHandle(_raw_stream(index))
  else:
    h = StreamHandle(torch.cuda.current_stream(index).cuda_stream)
  h.index = index
  return h


class PinnedWords:
  """Ring of pinned int32 words per device for asynchronous read-backs of device-side counts (visible gaussians,
  tile overlaps).  Every read-back takes the NEXT word, so a second projection / mapper front enqueued on the same
  stream before the first one's count has been consumed (pipelined views) cannot overwrite it; pinned allocations are
  made once per device (cudaHostAlloc is a millisecond-scale call)."""
  SLOTS = 64

  def __init__(self):
    self._rings = {}

  def take(self, device) -> torch.Tensor:
    key = (device.type, device.index)
    ring = self._rings.get(key)
    if ring is None:
      ring = self._rings[key] = [torch.zeros((self.SLOTS,), dtype=torch.int32).pin_memory(), 0]
    words, nxt = ring
    ring[1] = (nxt + 1) % self.SLOTS
    return words[nxt:nxt + 1]


pinned_words = PinnedWords()


def workspace(nbytes: int, device) -> torch.Tensor:
  return torch.empty((max(int(nbytes), 16),), dtype=torch.uint8, device=device)
