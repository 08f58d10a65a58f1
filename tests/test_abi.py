"""The drop-in boundary: libgsplat_b200.so loads and exports every symbol include/gsplat_b200.h declares.
No compute call is made here (no GPU in the CPU suite)."""
import ctypes
import re
from pathlib import Path

from taichi_gaussian_rasterizer_b200 import _native

ROOT = Path(__file__).resolve().parents[1]


def declared_symbols():
  text = (ROOT / "include" / "gsplat_b200.h").read_text()
  text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
  return sorted(set(re.findall(r"\b(gs_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_the_path():
  names = declared_symbols()
  for required in ("gs_project_fwd", "gs_project_bwd", "gs_sh_fwd", "gs_sh_bwd", "gs_tile_count",
                   "gs_full_cumsum", "gs_tile_emit_keys", "gs_radix_sort_pairs", "gs_find_ranges",
                   "gs_raster_fwd", "gs_raster_bwd", "gs_last_error_string"):
    assert required in names


def test_library_exports_every_declared_symbol():
  lib = ctypes.CDLL(str(_native.LIB_PATH))
  missing = [n for n in declared_symbols() if not hasattr(lib, n)]
  assert not missing, f"declared in include/gsplat_b200.h but not exported: {missing}"
  assert sorted(_native.EXPORTS) == declared_symbols()


def test_abi_version_and_error_string():
  lib = _native.lib()
  assert lib.gs_abi_version() == 5
  assert isinstance(lib.gs_last_error_string(), bytes)


def test_struct_sizes_match_header():
  # natural alignment of the POD parameter blocks (checked against sizeof in the C++ build by layout)
  assert ctypes.sizeof(_native.GsProjectParams) == 64
  assert ctypes.sizeof(_native.GsSHParams) == 40
  assert ctypes.sizeof(_native.GsTileParams) == 32
  assert ctypes.sizeof(_native.GsRasterParams) == 112


def test_invalid_arguments_return_errors_not_crashes():
  lib = _native.lib()
  rc = lib.gs_raster_fwd(None, None, None, None, None, None, None, None, None, ctypes.c_size_t(0), None)
  assert rc == -1
  assert b"null params" in lib.gs_last_error_string()
  p = _native.GsRasterParams(dtype=0, image_width=16, image_height=16, tile_size=12, num_features=3,
                             pixel_stride_x=2, pixel_stride_y=2)
  rc = lib.gs_raster_fwd(ctypes.byref(p), None, None, None, None, None, None, None, None, ctypes.c_size_t(0), None)
  assert rc == -2 and b"tile_size" in lib.gs_last_error_string()
  p = _native.GsRasterParams(dtype=0, image_width=16, image_height=16, tile_size=16, num_features=3,
                             pixel_stride_x=1, pixel_stride_y=1, kernel_variant=1)
  rc = lib.gs_raster_fwd(ctypes.byref(p), None, None, None, None, None, None, None, None, ctypes.c_size_t(0), None)
  assert rc == -1 and b"kernel_variant" in lib.gs_last_error_string()
  rc = lib.gs_raster_bwd(ctypes.byref(p), None, None, None, None, None, None, None, None, None, None,
                         ctypes.c_size_t(0), None)
  assert rc == -1 and b"kernel_variant" in lib.gs_last_error_string()
  rc = lib.gs_radix_sort_pairs(ctypes.c_int64(10), ctypes.c_int32(3), None, None, None, None, 0, 8, None,
                               ctypes.c_size_t(0), None)
  assert rc == -1


def test_sh_bwd_rejects_accumulate_params():
  """GsSHParams.accumulate_params only selects add / overwrite for gs_sh_bwd_flush; gs_sh_bwd reserves it."""
  lib = _native.lib()
  p = _native.GsSHParams(_native.GS_F32, 3, 16, 1, 100, 50, 1, 0)
  rc = lib.gs_sh_bwd(ctypes.byref(p), None, None, None, None, None, None, None, None, None)
  assert rc == -1 and b"accumulate_params" in lib.gs_last_error_string()


def test_missing_cuda_tensor_fails_loudly():
  import pytest
  import torch
  from taichi_gaussian_rasterizer_b200 import RasterConfig, map_to_tiles
  with pytest.raises(RuntimeError, match="no CPU path"):
    map_to_tiles(torch.rand(4, 7), torch.rand(4, 1), (32, 32), RasterConfig())
