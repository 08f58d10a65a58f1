"""Spherical harmonics of every degree 0..3 on the batched, deferred and counted paths: the shapes the C entry points
accept, the predicate that routes tensors to them, and the row bounds of a sliced deferred flush.  No compute call is
made here (no GPU in the CPU suite): the calls below return before any CUDA work."""
import ctypes

import pytest
import torch

from taichi_gaussian_rasterizer_b200 import _native
from taichi_gaussian_rasterizer_b200.distributed import GradientBucket
from taichi_gaussian_rasterizer_b200.grad_sinks import DeferredSH
from taichi_gaussian_rasterizer_b200.spherical_harmonics import sh_fast_path

GS_OK, GS_ERR_UNSUPPORTED = 0, -2


def _views(lib, p, num_views):
  arr = ctypes.c_void_p * max(num_views, 1)
  return lib.gs_sh_fwd_views(ctypes.byref(p), ctypes.c_int32(num_views), None, None, arr(), arr(), None)


def _flush(lib, p, num_views):
  arr = ctypes.c_void_p * max(num_views, 1)
  return lib.gs_sh_bwd_flush(ctypes.byref(p), ctypes.c_int32(num_views), arr(), arr(), None, None, None)


@pytest.mark.parametrize("d", [1, 4, 9, 16])
def test_batched_entry_points_accept_every_degree(d):
  """gs_sh_fwd_views and gs_sh_bwd_flush take D = 1, 4, 9, 16 (f32, K = 3); with no views or no points there is
  nothing to do and they return GS_OK."""
  lib = _native.lib()
  empty = _native.GsSHParams(_native.GS_F32, 3, d, 1, 0, 0, 0, 1)
  some = _native.GsSHParams(_native.GS_F32, 3, d, 1, 1000, 0, 1, 1)   # accumulate: zero views leave the rows alone
  assert _views(lib, empty, 4) == GS_OK, lib.gs_last_error_string()
  assert _views(lib, some, 0) == GS_OK, lib.gs_last_error_string()
  assert _flush(lib, empty, 4) == GS_OK, lib.gs_last_error_string()
  assert _flush(lib, some, 0) == GS_OK, lib.gs_last_error_string()


@pytest.mark.parametrize("dtype,k,d", [(_native.GS_F32, 3, 25), (_native.GS_F32, 4, 16), (_native.GS_F32, 4, 9),
                                       (_native.GS_F64, 3, 16)])
def test_batched_entry_points_refuse_other_shapes(dtype, k, d):
  """Degree 4, K != 3 and f64 stay unsupported, with a message that names K and D."""
  lib = _native.lib()
  p = _native.GsSHParams(dtype, k, d, 1, 0, 0, 1, 1)
  for call in (_views, _flush):
    assert call(lib, p, 1) == GS_ERR_UNSUPPORTED
    msg = lib.gs_last_error_string()
    assert f"K = {k}".encode() in msg and f"D = {d}".encode() in msg, msg


def test_fast_path_predicate():
  """One predicate decides which SH tensors the batched / deferred / counted paths serve: f32, K = 3, degree 0..3."""
  for d in (1, 4, 9, 16):
    assert sh_fast_path(torch.zeros(5, 3, d))
  assert not sh_fast_path(torch.zeros(5, 3, 25))
  assert not sh_fast_path(torch.zeros(5, 4, 16))
  assert not sh_fast_path(torch.zeros(5, 3, 16, dtype=torch.float64))
  assert not sh_fast_path(torch.zeros(5, 48))


@pytest.mark.parametrize("d", [1, 4, 9, 16])
@pytest.mark.parametrize("n", [1, 3, 4999])
def test_flush_chunk_bounds_are_multiples_of_four_rows(n, d):
  """DeferredSH.flush(chunks=): the slices cover [0, n) in order without gaps, are non-empty, and every inner bound is
  a multiple of 4 rows, so a slice starts a multiple of 4 floats (16 B) into the sink at every row width 3 D."""
  row = 3 * d
  for chunks in (1, 2, 3, 4, 8):
    b = DeferredSH.chunk_bounds(n, chunks)
    assert b[0] == 0 and b[-1] == n and len(b) - 1 <= chunks
    assert all(lo < hi for lo, hi in zip(b, b[1:]))
    assert all(lo % 4 == 0 and (lo * row) % 4 == 0 for lo in b[:-1])


def test_odd_gaussian_count_puts_the_sh_slice_off_16_bytes():
  """Why the flush and the dense backward have 4 B-unit variants: in a bucket laid out [position, log_scaling,
  rotation, alpha_logit, feature] the feature slice starts 11 N floats in, 16 B aligned only when N % 4 == 0."""
  for n, aligned in ((3000, True), (3001, False), (4999, False)):
    params = [torch.zeros(n, 3, requires_grad=True), torch.zeros(n, 3, requires_grad=True),
              torch.zeros(n, 4, requires_grad=True), torch.zeros(n, requires_grad=True),
              torch.zeros(n, 3, 9, requires_grad=True)]
    bucket = GradientBucket(params)
    assert bucket.flat.data_ptr() % 16 == 0
    assert (params[4].grad.data_ptr() % 16 == 0) == aligned
    assert params[4].grad.data_ptr() % 4 == 0
