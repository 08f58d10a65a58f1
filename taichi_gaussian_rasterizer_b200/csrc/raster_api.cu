// raster_api.cu — gs_raster_fwd / gs_raster_bwd(_with_weight): validation and kernel-family selection.
#include "raster.cuh"

using namespace gs;

static int check_raster(const GsRasterParams* p, const char* who) {
  if (!p) { set_error("%s: null params", who); return GS_ERR_INVALID; }
  if (p->dtype != GS_F32 && p->dtype != GS_F64 && p->dtype != GS_BF16) {
    set_error("%s: dtype must be GS_F32, GS_F64 or GS_BF16", who);
    return GS_ERR_INVALID;
  }
  if (p->image_width <= 0 || p->image_height <= 0 || p->num_features <= 0 || p->num_points < 0 || p->num_overlaps < 0) {
    set_error("%s: bad sizes (image %dx%d, F=%d, V=%lld, K=%lld)", who, p->image_width, p->image_height,
              p->num_features, (long long)p->num_points, (long long)p->num_overlaps);
    return GS_ERR_INVALID;
  }
  if (p->tile_size != 8 && p->tile_size != 16 && p->tile_size != 32) {
    set_error("%s: tile_size must be 8, 16 or 32, got %d", who, p->tile_size);
    return GS_ERR_UNSUPPORTED;
  }
  if (p->kernel_variant != 0) {
    set_error("%s: kernel_variant is reserved and must be 0, got %d", who, p->kernel_variant);
    return GS_ERR_INVALID;
  }
  const int sx = p->pixel_stride_x, sy = p->pixel_stride_y;
  if (sx <= 0 || sy <= 0 || (p->tile_size * p->tile_size) / (sx * sy) < 32) {  // rasterizer/backward.py:33-34
    set_error("%s: pixel_stride (%d, %d) and tile_size %d must allow at least one warp sized (32) tile", who, sx, sy,
              p->tile_size);
    return GS_ERR_INVALID;
  }
  if (p->dtype == GS_BF16) {   // bf16 feature storage exists on the fast kernels only (raster_fast_supported)
    const char* why = p->num_features < 8 || p->num_features > 256 ? "8..256 feature channels"
                      : p->tile_size != 16                          ? "tile_size 16"
                      : !p->use_alpha_blending                      ? "alpha blending"
                      : p->antialias                                ? "no antialiasing"
                      : p->num_points >= (1ll << 31)                ? "fewer than 2^31 gaussians"
                                                                    : nullptr;
    if (why) {
      set_error("%s: GS_BF16 features need %s (F=%d, tile_size %d, alpha blending %d, antialias %d)", who, why,
                p->num_features, p->tile_size, p->use_alpha_blending, p->antialias);
      return GS_ERR_UNSUPPORTED;
    }
  }
  return GS_OK;
}

extern "C" {

size_t gs_raster_workspace_bytes(const GsRasterParams* p) {
  if (!p) return 0;
  return raster_fast_supported(*p) ? raster_fast_workspace_bytes(*p) : 0;
}

int gs_raster_fwd(const GsRasterParams* p, const void* gaussians2d, const void* features, const int32_t* tile_ranges,
                  const int32_t* overlap_to_point, void* image, void* image_alpha, void* visibility, void* workspace,
                  size_t workspace_bytes, void* stream) {
  int rc = check_raster(p, "gs_raster_fwd");
  if (rc != GS_OK) return rc;
  GS_CHECK_ARG(tile_ranges && image && image_alpha, "gs_raster_fwd: null tensor");
  GS_CHECK_ARG(p->num_points == 0 || (gaussians2d && features), "gs_raster_fwd: null gaussians / features");
  GS_CHECK_ARG(p->num_overlaps == 0 || overlap_to_point, "gs_raster_fwd: null overlap_to_point");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t es = p->dtype == GS_F64 ? 8 : 4;   // GS_BF16: visibility / gradients are f32
  if (p->compute_visibility && visibility && p->num_points > 0)
    GS_CUDA(cudaMemsetAsync(visibility, 0, (size_t)p->num_points * es, st));
  RasterArgs a = {};
  a.gaussians2d = gaussians2d; a.features = features; a.tile_ranges = tile_ranges;
  a.overlap_to_point = overlap_to_point; a.image = image; a.image_alpha = image_alpha; a.visibility = visibility;
  a.workspace = workspace; a.workspace_bytes = workspace_bytes;
  if (raster_fast_supported(*p)) {
    const size_t need = raster_fast_workspace_bytes(*p);
    if (workspace == nullptr || workspace_bytes < need) {
      set_error("gs_raster_fwd: workspace %zu < %zu bytes", workspace_bytes, need);
      return GS_ERR_WORKSPACE;
    }
    return raster_fwd_fast(*p, a, st);
  }
  return raster_fwd_generic(*p, a, st);
}

int gs_raster_bwd_with_weight(const GsRasterParams* p, const void* gaussians2d, const void* features,
                              const int32_t* tile_ranges, const int32_t* overlap_to_point, const void* image,
                              const void* grad_image, const void* image_weight, const void* grad_image_weight,
                              void* grad_gaussians, void* grad_features, void* point_heuristic, void* workspace,
                              size_t workspace_bytes, void* stream) {
  int rc = check_raster(p, "gs_raster_bwd");
  if (rc != GS_OK) return rc;
  GS_CHECK_ARG(tile_ranges && grad_image && (image || !p->use_alpha_blending), "gs_raster_bwd: null tensor");
  GS_CHECK_ARG(p->num_points == 0 || (gaussians2d && features), "gs_raster_bwd: null gaussians / features");
  GS_CHECK_ARG(p->num_overlaps == 0 || overlap_to_point, "gs_raster_bwd: null overlap_to_point");
  // quantile mode: the weight is W > 0, piecewise constant, so its gradient contributes nothing
  if (!p->use_alpha_blending) grad_image_weight = nullptr;
  GS_CHECK_ARG(!grad_image_weight || image_weight, "gs_raster_bwd_with_weight: grad_image_weight without image_weight");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t es = p->dtype == GS_F64 ? 8 : 4;   // GS_BF16: visibility / gradients are f32
  if (grad_gaussians && p->num_points > 0) GS_CUDA(cudaMemsetAsync(grad_gaussians, 0, (size_t)p->num_points * 7 * es, st));
  if (grad_features && p->num_points > 0)
    GS_CUDA(cudaMemsetAsync(grad_features, 0, (size_t)p->num_points * p->num_features * es, st));
  RasterArgs a = {};
  a.gaussians2d = gaussians2d; a.features = features; a.tile_ranges = tile_ranges;
  a.overlap_to_point = overlap_to_point; a.image_in = image; a.grad_image = grad_image;
  a.image_weight = grad_image_weight ? image_weight : nullptr; a.grad_image_weight = grad_image_weight;
  a.grad_gaussians = grad_gaussians; a.grad_features = grad_features; a.point_heuristic = point_heuristic;
  a.workspace = workspace; a.workspace_bytes = workspace_bytes;
  if (raster_fast_supported(*p)) {
    const size_t need = raster_fast_workspace_bytes(*p);
    if (workspace == nullptr || workspace_bytes < need) {
      set_error("gs_raster_bwd: workspace %zu < %zu bytes", workspace_bytes, need);
      return GS_ERR_WORKSPACE;
    }
    return raster_bwd_fast(*p, a, st);
  }
  return raster_bwd_generic(*p, a, st);
}

int gs_raster_bwd(const GsRasterParams* p, const void* gaussians2d, const void* features, const int32_t* tile_ranges,
                  const int32_t* overlap_to_point, const void* image, const void* grad_image, void* grad_gaussians,
                  void* grad_features, void* point_heuristic, void* workspace, size_t workspace_bytes, void* stream) {
  return gs_raster_bwd_with_weight(p, gaussians2d, features, tile_ranges, overlap_to_point, image, grad_image, nullptr,
                                   nullptr, grad_gaussians, grad_features, point_heuristic, workspace, workspace_bytes,
                                   stream);
}

}  // extern "C"
