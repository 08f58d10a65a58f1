// raster.cuh — internal interface between the rasterizer entry points (raster_api.cu) and the
// kernel families: raster_generic.cu (every dtype / mode, fidelity first; also the f64 gradcheck
// path) and raster_fast_fwd.cu / raster_fast_bwd.cu / raster_fast_bwd_wide.cu (f32, alpha blending, tile 16: the
// measured path).
#pragma once

#include "common.cuh"

namespace gs {

struct RasterArgs {
  const void* gaussians2d;
  const void* features;
  const int32_t* tile_ranges;
  const int32_t* overlap_to_point;
  // forward
  void* image;
  void* image_alpha;
  void* visibility;
  // backward
  const void* image_in;
  const void* grad_image;
  const void* image_weight;        // (H, W) forward image_alpha; with grad_image_weight: the weight's gradient too
  const void* grad_image_weight;   // (H, W) or NULL (no weight gradient: the kernels of gs_raster_bwd)
  void* grad_gaussians;
  void* grad_features;
  void* point_heuristic;
  void* workspace;
  size_t workspace_bytes;
};

inline int tiles_wide(const GsRasterParams& p) { return (p.image_width + p.tile_size - 1) / p.tile_size; }
inline int tiles_high(const GsRasterParams& p) { return (p.image_height + p.tile_size - 1) / p.tile_size; }

int raster_fwd_generic(const GsRasterParams& p, const RasterArgs& a, cudaStream_t st);
int raster_bwd_generic(const GsRasterParams& p, const RasterArgs& a, cudaStream_t st);

bool raster_fast_supported(const GsRasterParams& p);
size_t raster_fast_workspace_bytes(const GsRasterParams& p);
int raster_fwd_fast(const GsRasterParams& p, const RasterArgs& a, cudaStream_t st);
int raster_bwd_fast(const GsRasterParams& p, const RasterArgs& a, cudaStream_t st);

}  // namespace gs
