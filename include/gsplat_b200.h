/*
 * gsplat_b200.h — C ABI of libgsplat_b200.so: the sm_100a implementation of the
 * taichi_splatting render path (project -> SH -> tile map -> sort -> rasterize fwd/bwd).
 *
 * This is the drop-in boundary.  The reference's native boundary is only the three CUB
 * wrappers of taichi_splatting/cuda_lib/module.cpp:14-18; its other kernels are Taichi-JIT
 * and have no ABI, so each entry point below cites the reference kernel / wrapper it
 * replaces.  Paths are relative to /root/reference/taichi_splatting/.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless stated;
 *   - the caller owns all memory (inputs, outputs, workspaces); the library never allocates
 *     device memory and keeps no pointer after returning;
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no call synchronises
 *     the host; calls are re-entrant;
 *   - return value: GS_OK (0) or a negative GsStatus; gs_last_error_string() describes the last
 *     failure on the calling thread.  Nothing throws or exits across this boundary;
 *   - `dtype` selects float (GS_F32) or double (GS_F64) for every `void*` floating tensor of
 *     the call; the tile mapper is f32 only, like the reference (mapper/tile_mapper.py:12); GS_BF16 is valid in
 *     GsRasterParams.dtype only and selects bfloat16 for the feature side of the rasterizer (see there);
 *   - tensors are dense row-major with the shapes stated.
 */
#ifndef GSPLAT_B200_H
#define GSPLAT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum GsStatus {
  GS_OK = 0,
  GS_ERR_INVALID = -1,     /* bad argument / shape */
  GS_ERR_UNSUPPORTED = -2, /* configuration outside the implemented set */
  GS_ERR_CUDA = -3,        /* a CUDA runtime call failed */
  GS_ERR_WORKSPACE = -4    /* workspace too small */
} GsStatus;

typedef enum GsDtype { GS_F32 = 0, GS_F64 = 1, GS_BF16 = 2 } GsDtype;

int gs_abi_version(void);
const char* gs_last_error_string(void);

/* ------------------------------------------------------------------ projection
 * replaces project_kernel + torch.nonzero + gather (perspective/projection.py:31-80, :146-149)
 * and indexed_project_kernel.grad (:83-118, :164-185). */
typedef struct GsProjectParams {
  int32_t dtype;
  int32_t image_width, image_height;
  int32_t accumulate_grads; /* gs_project_bwd: ADD the per gaussian gradients of the visible rows into the caller's
                               buffers (gradient bucket of a multi-view batch) instead of writing them dense */
  int64_t num_points;      /* N */
  double near_plane, far_plane;
  double blur_cov, clamp_margin, alpha_threshold;
} GsProjectParams;

size_t gs_project_fwd_workspace_bytes(const GsProjectParams* p);

/* position (N,3) log_scaling (N,3) rotation (N,4 xyzw) alpha_logit (N,1) T_camera_world (4,4)
 * projection (4: fx fy cx cy).  Outputs have capacity N; the first *num_visible rows are
 * valid, in ascending gaussian index order (identical to nonzero()):
 * points (N,7) depth (N,1) indexes (N) int64, num_visible: one int32 on the device. */
int gs_project_fwd(const GsProjectParams* p, const void* position, const void* log_scaling,
                   const void* rotation, const void* alpha_logit, const void* T_camera_world,
                   const void* projection, void* points, void* depth, int64_t* indexes,
                   int32_t* num_visible, void* workspace, size_t workspace_bytes, void* stream);

/* grad_points (V,7) grad_depth (V,1) -> dense grads, fully written (zero for culled points):
 * grad_position (N,3) grad_log_scaling (N,3) grad_rotation (N,4) grad_alpha_logit (N,1)
 * grad_T_camera_world (4,4; last row zero) grad_projection (4).  Any grad pointer may be NULL.
 * With p->accumulate_grads the four per gaussian buffers are NOT cleared: the rows of the visible gaussians are
 * incremented, all other rows are left as they are (`indexes` must be unique, as the visible set is). */
int gs_project_bwd(const GsProjectParams* p, int64_t num_visible, const void* position,
                   const void* log_scaling, const void* rotation, const void* alpha_logit,
                   const void* T_camera_world, const void* projection, const int64_t* indexes,
                   const void* grad_points, const void* grad_depth, void* grad_position,
                   void* grad_log_scaling, void* grad_rotation, void* grad_alpha_logit,
                   void* grad_T_camera_world, void* grad_projection, void* stream);
/* Same with the visible count still on the device: grad_points / grad_depth / indexes have `capacity` rows, the first
 * *count_dev of them are used (the capacity-sized outputs of gs_project_fwd, handed on without reading num_visible
 * back: the reference reads it with torch.nonzero, projection.py:146-149 — a device synchronisation per view). */
int gs_project_bwd_counted(const GsProjectParams* p, int64_t capacity, const int32_t* count_dev, const void* position,
                           const void* log_scaling, const void* rotation, const void* alpha_logit,
                           const void* T_camera_world, const void* projection, const int64_t* indexes,
                           const void* grad_points, const void* grad_depth, void* grad_position,
                           void* grad_log_scaling, void* grad_rotation, void* grad_alpha_logit,
                           void* grad_T_camera_world, void* grad_projection, void* stream);

/* ------------------------------------------------------------------ spherical harmonics
 * replaces evaluate_sh_at_kernel and its .grad (spherical_harmonics.py:118-134, :154-161). */
typedef struct GsSHParams {
  int32_t dtype;
  int32_t num_channels;    /* K */
  int32_t num_coeffs;      /* D = (degree+1)^2, degree 0..3 */
  int32_t indexes_sorted_unique; /* hint: indexes strictly ascending (the visible set of gs_project_fwd); lets
                                    gs_sh_bwd write dense gradient rows without atomics.  0 = no assumption. */
  int64_t num_points;      /* M */
  int64_t num_indexes;     /* V */
  int32_t accumulate_params; /* gs_sh_bwd_flush: 1 = add the sum to grad_params, 0 = overwrite the rows with it.
                                gs_sh_bwd: reserved, must be 0 (GS_ERR_INVALID otherwise). */
  int32_t params_is_forward_output; /* gs_sh_bwd: the `params` argument holds the forward OUTPUT (V,K) instead of the
                                       coefficients — enough for grad_params (the coefficients only enter through the
                                       clamp mask, and v in (0,1) <=> clamp(v) in (0,1)) and 4KD bytes per gaussian
                                       less traffic; dense path only, grad_positions / grad_camera_pos must be NULL */
} GsSHParams;

/* params (M,K,D) positions (M,3) indexes (V) int64 camera_pos (3) -> out (V,K) */
int gs_sh_fwd(const GsSHParams* p, const void* params, const void* positions,
              const int64_t* indexes, const void* camera_pos, void* out, void* stream);

/* Same, but the number of valid indexes is still on the device (count_dev, one int32, e.g. num_visible of
 * gs_project_fwd): p->num_indexes is the CAPACITY of indexes / out, rows >= *count_dev are left untouched.  Lets the
 * caller enqueue the SH evaluation before it reads the visible count back. */
int gs_sh_fwd_counted(const GsSHParams* p, const void* params, const void* positions,
                      const int64_t* indexes, const void* camera_pos, const int32_t* count_dev,
                      void* out, void* stream);

/* grad_out (V,K) -> grad_params (M,K,D) grad_positions (M,3) grad_camera_pos (3); each fully
 * written (zeroed then accumulated; repeated indexes are summed).  Any may be NULL.  With p->indexes_sorted_unique,
 * f32, K = 3 and D in {1, 4, 9, 16} the rows are written densely without atomics (16 B units at D = 4, 16 when the
 * pointers are 16 B aligned, 4 B units otherwise); every other shape takes the generic atomic kernel. */
int gs_sh_bwd(const GsSHParams* p, const void* params, const void* positions,
              const int64_t* indexes, const void* camera_pos, const void* grad_out,
              void* grad_params, void* grad_positions, void* grad_camera_pos, void* stream);

/* Deferred coefficient gradient for a multi-view batch (f32, K = 3, D in {1, 4, 9, 16}; any other shape returns
 * GS_ERR_UNSUPPORTED).  evaluate_sh_at_kernel.grad
 * (spherical_harmonics.py:154-161) followed by autograd's accumulation rewrites the whole (M,K,D) gradient once per
 * view; the coefficient gradient of a view is the outer product of the masked colour gradient with the basis of the
 * viewing direction, so a view only has to keep K floats per gaussian:
 *   gs_sh_bwd_stage: staged (M,K) <- grad_out (V,K) scattered by `indexes`, zero where the forward value
 *                    (forward_out (V,K), the clamped output of gs_sh_fwd) sits on the clamp and where culled;
 *   gs_sh_bwd_flush: grad_params (M,K,D) += sum over the num_views staged views of staged_v (x) basis(positions -
 *                    camera_positions[v]); `staged` / `camera_positions` are HOST arrays of num_views device pointers
 *                    ((M,K) and (3,) floats), num_views <= GS_SH_MAX_DEFERRED_VIEWS.  With p->accumulate_params = 0
 *                    the rows are OVERWRITTEN with the sum (zeroed when num_views = 0): the first flush of a batch
 *                    then needs neither a zero fill of grad_params before nor a read of it.
 * p->num_points = M, p->num_indexes = V (stage only).  grad_params may sit at any 4 B aligned address (a slice of a
 * flat gradient bucket): the flush moves 16 B units only when grad_params is 16 B aligned, 4 B units otherwise. */
#define GS_SH_MAX_DEFERRED_VIEWS 16
int gs_sh_bwd_stage(const GsSHParams* p, const void* forward_out, const int64_t* indexes, const void* grad_out,
                    void* staged, void* stream);
/* gs_sh_bwd_stage with the number of indexes still on the device (p->num_indexes = capacity of indexes / forward_out /
 * grad_out; `staged` is always cleared first). */
int gs_sh_bwd_stage_counted(const GsSHParams* p, const void* forward_out, const int64_t* indexes, const void* grad_out,
                            const int32_t* count_dev, void* staged, void* stream);
int gs_sh_bwd_flush(const GsSHParams* p, int32_t num_views, const void* const* staged,
                    const void* const* camera_positions, const void* positions, void* grad_params, void* stream);

/* Batched evaluation for the views of a multi-view batch (f32, K = 3, D in {1, 4, 9, 16}): evaluate_sh_at_kernel
 * (spherical_harmonics.py:118-134) reads the 4 K D byte coefficient row of every visible gaussian once per VIEW;
 * gs_sh_fwd_views reads every row once per BATCH and writes one dense colour tensor (M,K) per view (outs /
 * camera_positions: HOST arrays of num_views device pointers, num_views <= GS_SH_MAX_DEFERRED_VIEWS; same arithmetic
 * and clamp as gs_sh_fwd).  A view then takes its visible rows with gs_gather_rows_counted: out[j] = src[indexes[j]]
 * for j < *count_dev (count_dev NULL: j < capacity), rows of row_floats = 3 floats — the count may still be on the
 * device, as for gs_sh_fwd_counted.  params is read in 16 B units only at D = 4, 16 and when 16 B aligned. */
int gs_sh_fwd_views(const GsSHParams* p, int32_t num_views, const void* params, const void* positions,
                    const void* const* camera_positions, void* const* outs, void* stream);
int gs_gather_rows_counted(int64_t capacity, int32_t row_floats, const void* src, const int64_t* indexes,
                           const int32_t* count_dev, void* out, void* stream);

/* Plain (non-SH) features of the visible set: replaces `features = gaussians.feature[indexes]` of render_gaussians
 * (renderer.py:152-153) and the index_put of its backward.  Rows of row_floats f32, any width; the gathered rows may
 * land inside wider rows (out_stride / out_offset, in floats: e.g. behind the two depth channels of render_depth);
 * `indexes` are unique (the visible set), so the scatter writes without atomics after zero-filling dst (dst_rows rows).
 * count_dev (optional): the number of valid indexes still on the device, capacity = rows of `indexes`. */
int gs_gather_rows_strided(int64_t capacity, int32_t row_floats, const float* src, const int64_t* indexes,
                           const int32_t* count_dev, float* out, int32_t out_stride, int32_t out_offset, void* stream);
int gs_scatter_rows_strided(int64_t capacity, int32_t row_floats, const float* src, int32_t src_stride,
                            int32_t src_offset, const int64_t* indexes, const int32_t* count_dev, int64_t dst_rows,
                            float* dst, void* stream);
/* The same two for rows of 2-byte elements (bfloat16 features of a GS_BF16 rasterization; the bits are copied):
 * row_elems, out_stride / out_offset and src_stride / src_offset count 2-byte elements. */
int gs_gather_rows_strided_u16(int64_t capacity, int32_t row_elems, const uint16_t* src, const int64_t* indexes,
                               const int32_t* count_dev, uint16_t* out, int32_t out_stride, int32_t out_offset,
                               void* stream);
int gs_scatter_rows_strided_u16(int64_t capacity, int32_t row_elems, const uint16_t* src, int32_t src_stride,
                                int32_t src_offset, const int64_t* indexes, const int32_t* count_dev, int64_t dst_rows,
                                uint16_t* dst, void* stream);

/* render_depth: the rendered (P, channels) image split into its first `split` channels (depth, depth^2) and the rest,
 * and the inverse for the backward (a NULL part stands for zeros) — replaces the two strided slices of
 * renderer.py:215-222 and autograd's zero-padded slice backward of each.  f32, contiguous rows. */
int gs_split_channels(int64_t rows, int32_t channels, int32_t split, const float* src, float* first, float* rest,
                      void* stream);
int gs_merge_channels(int64_t rows, int32_t channels, int32_t split, const float* first, const float* rest, float* dst,
                      void* stream);

/* ------------------------------------------------------------------ tile mapper (f32)
 * replaces tile_overlaps_kernel / generate_sort_keys_kernel / find_ranges_kernel
 * (mapper/tile_mapper.py:73-84, :112-144, :90-110) with the OBB query of
 * taichi_lib/grid_query.py:9-91, and cuda_lib.full_cumsum / cuda_lib.radix_sort_pairs
 * (cuda_lib/full_cumsum.cu:16-67, cuda_lib/radix_sort_pairs.cu:9-69). */
typedef struct GsTileParams {
  int32_t image_width, image_height; /* unpadded; padded to tile_size internally */
  int32_t tile_size;
  int32_t use_depth16;               /* 0: u64 key = tile<<32 | f32 bits; 1: u32 key = tile<<16 | depth16 */
  int64_t num_points;                /* V */
  double alpha_threshold;
} GsTileParams;

/* gaussians (V,7) -> counts (V) int32 */
int gs_tile_count(const GsTileParams* p, const float* gaussians, int32_t* counts, void* stream);

/* full_cumsum: out has n+1 entries, out[i] = sum(in[0..i)), out[n] = total (stays on the device;
 * the caller reads it back when it needs the size).  elem_bytes 4 (int32) or 8 (int64). */
size_t gs_full_cumsum_workspace_bytes(int64_t n, int32_t elem_bytes);
int gs_full_cumsum(int64_t n, int32_t elem_bytes, const void* in, void* out, void* workspace,
                   size_t workspace_bytes, void* stream);
/* Same over the first *count_dev of `capacity` elements (count on the device; the rest scan as zeros): out[i] for
 * i <= *count_dev as above, and the total also at total_out (one element, a fixed address the host can copy back
 * without knowing the count). */
int gs_full_cumsum_counted(int64_t capacity, int32_t elem_bytes, const int32_t* count_dev, const void* in, void* out,
                           void* total_out, void* workspace, size_t workspace_bytes, void* stream);

/* gaussians (V,7) depth (V) cum (V) -> keys (K) u64|u32, values (K) int32 (gaussian index) */
int gs_tile_emit_keys(const GsTileParams* p, const float* gaussians, const float* depth,
                      const int32_t* cum, void* keys, int32_t* values, void* stream);

/* stable LSD onesweep radix sort of (key, int32 value) pairs on key bits [begin_bit, end_bit).
 * key_bytes 4 or 8.  Inputs are preserved. */
size_t gs_radix_sort_pairs_workspace_bytes(int64_t n, int32_t key_bytes, int32_t begin_bit,
                                           int32_t end_bit);
int gs_radix_sort_pairs(int64_t n, int32_t key_bytes, const void* keys_in, const int32_t* values_in,
                        void* keys_out, int32_t* values_out, int32_t begin_bit, int32_t end_bit,
                        void* workspace, size_t workspace_bytes, void* stream);
/* Same for the first *count_dev of `capacity` pairs (count on the device; workspace sized for `capacity`; output rows
 * >= *count_dev are left untouched). */
int gs_radix_sort_pairs_counted(int64_t capacity, const int32_t* count_dev, int32_t key_bytes, const void* keys_in,
                                const int32_t* values_in, void* keys_out, int32_t* values_out, int32_t begin_bit,
                                int32_t end_bit, void* workspace, size_t workspace_bytes, void* stream);

/* sorted keys (K) -> tile_ranges (T,2) int32, fully written ([0,0] for empty tiles) */
int gs_find_ranges(const GsTileParams* p, int64_t num_overlaps, const void* sorted_keys,
                   int32_t* tile_ranges, void* stream);

/* Depth-first tile mapping: produces exactly the overlap_to_point / tile_ranges of
 * count -> emit_keys -> sort(32 + tile bits) -> find_ranges (mapper/tile_mapper.py:146-196) with a third of the sort
 * traffic: (1) gs_depth_keys: u32 depth key (f32 bits, or depth16) + index per gaussian; sort them (stable) to get
 * `perm`; (2) gs_tile_count_perm / gs_tile_emit_tiles visit the gaussians in that order and emit bare tile ids;
 * (3) a stable sort on the tile id bits only; (4) gs_find_ranges_tiles.  perm (V) int32, tile_ids (K) u32. */
/* near_plane > 0: `depth` is linear camera depth and the key is built from its NDC value
 * 1 - (1/d - 1/far) / (1/near - 1/far) (torch_lib/projection.py:120-123), evaluated with the same f32 operation
 * sequence as torch's eager CUDA kernels; near_plane <= 0: `depth` already is the sort depth. */
int gs_depth_keys(const GsTileParams* p, const float* depth, double near_plane, double far_plane,
                  uint32_t* keys, int32_t* values, void* stream);
/* Same with the number of gaussians still on the device (count_dev, e.g. num_visible of gs_project_fwd):
 * p->num_points is the CAPACITY of depth / keys / values, rows >= *count_dev are left untouched.  Together with
 * gs_radix_sort_pairs_counted the depth ordering of a frame can be enqueued before the host reads the visible count. */
int gs_depth_keys_counted(const GsTileParams* p, const float* depth, double near_plane, double far_plane,
                          const int32_t* count_dev, uint32_t* keys, int32_t* values, void* stream);
/* tile_masks (V) uint64, optional (NULL = none) in both calls: the count pass records per slot which tiles of a span of
 * at most 32 tiles passed the test, the emit pass then expands those bits instead of repeating the OBB query and the
 * tile tests (spans above 32 tiles are flagged and recomputed).  Same outputs either way. */
int gs_tile_count_perm(const GsTileParams* p, const float* gaussians, const int32_t* perm, int32_t* counts,
                       uint64_t* tile_masks, void* stream);
/* Same with the number of gaussians still on the device (p->num_points = capacity of perm / counts / tile_masks). */
int gs_tile_count_perm_counted(const GsTileParams* p, const float* gaussians, const int32_t* perm,
                               const int32_t* count_dev, int32_t* counts, uint64_t* tile_masks, void* stream);
int gs_tile_emit_tiles(const GsTileParams* p, const float* gaussians, const int32_t* perm, const int32_t* cum,
                       const uint64_t* tile_masks, uint32_t* tile_ids, int32_t* values, void* stream);
int gs_find_ranges_tiles(const GsTileParams* p, int64_t num_overlaps, const uint32_t* sorted_tile_ids,
                         int32_t* tile_ranges, void* stream);
/* Capacity-bounded tail of the tile mapping: the overlap total K stays on the device (the int32 behind the scan's
 * total_out), tile_ids / values have `capacity` rows.  No host read-back anywhere in map_to_tiles, so a whole
 * forward + backward step can be captured in a CUDA graph (the reference synchronises the device twice here,
 * cuda_lib/full_cumsum.cu:45, radix_sort_pairs.cu:27).  Overlaps that would land at or beyond `capacity` are dropped
 * (the caller compares K with the capacity after the fact); gs_radix_sort_pairs_counted sorts min(K, capacity) rows. */
int gs_tile_emit_tiles_capped(const GsTileParams* p, const float* gaussians, const int32_t* perm, const int32_t* cum,
                              const uint64_t* tile_masks, int64_t capacity, uint32_t* tile_ids, int32_t* values,
                              void* stream);
/* ... and with the number of gaussians still on the device as well (p->num_points = capacity of perm / cum /
 * tile_masks, as left by gs_tile_count_perm_counted + gs_full_cumsum_counted): with this, gs_project_bwd_counted and
 * gs_sh_bwd_stage_counted a whole 3D view (render_gaussians forward + backward) runs without a host read-back. */
int gs_tile_emit_tiles_capped_counted(const GsTileParams* p, const float* gaussians, const int32_t* perm,
                                      const int32_t* cum, const uint64_t* tile_masks, const int32_t* count_dev,
                                      int64_t capacity, uint32_t* tile_ids, int32_t* values, void* stream);
int gs_find_ranges_tiles_counted(const GsTileParams* p, int64_t capacity, const int32_t* num_overlaps_dev,
                                 const uint32_t* sorted_tile_ids, int32_t* tile_ranges, void* stream);

/* ------------------------------------------------------------------ rasterizer
 * replaces _forward_kernel (rasterizer/forward.py:24-137) and _backward_kernel
 * (rasterizer/backward.py:52-228). */
typedef struct GsRasterParams {
  int32_t dtype;
  int32_t image_width, image_height;
  int32_t tile_size;                 /* 8, 16 or 32 */
  int32_t num_features;              /* F: 1..256 in f32 with tile_size 16, alpha blending and no antialiasing
                                        (antialiased: 1..7; 65..256 read rows of 16-byte aligned features in place
                                        when F is a multiple of 64); 1..40 in f32 otherwise (tile_size 32: 1..8);
                                        1..8 in f64 (tile_size 32: 1..4); 8..256 in bf16, see below.
                                        Other counts: GS_ERR_UNSUPPORTED */
  int32_t antialias;
  int32_t use_alpha_blending;
  int32_t compute_visibility;
  int32_t compute_point_heuristic;
  int32_t points_requires_grad, features_requires_grad;
  int32_t emulate_stale_tail;        /* reproduce forward.py:88 (SURVEY Q1); 1 for reference parity */
  int32_t pixel_stride_x, pixel_stride_y; /* validated like backward.py:33-34, otherwise a hint */
  int32_t workspace_holds_packed;    /* bwd: the workspace is untouched since a gs_raster_fwd call made with the same
                                        gaussians / features AND a requires_grad flag set (fwd then packs the
                                        backward records too); 0 = repack */
  int32_t kernel_variant;            /* reserved, must be 0 (GS_ERR_INVALID otherwise) */
  int64_t num_points;                /* V */
  int64_t num_overlaps;              /* K */
  double clamp_max_alpha, alpha_threshold, saturate_threshold;
  /* forward stops a tile once every pixel's transmittance 1-W is <= this; 0 = exact
   * (1-W == 0, after which no output can change).  The reference has no forward exit. */
  double forward_exit_transmittance;
} GsRasterParams;
/* dtype GS_BF16: bfloat16 storage of the feature side, f32 arithmetic.  features (V,F), image (H,W,F) and grad_image
 * (H,W,F) are bfloat16 (the image is the f32 blend rounded to nearest once); gaussians2d, image_alpha, visibility,
 * point_heuristic, grad_gaussians, image_weight and grad_image_weight are f32, and so is grad_features (V,F): it is
 * accumulated with f32 atomics, the caller rounds it or keeps it as an f32 master gradient.  Supported with F in
 * 8..256, tile_size 16, alpha blending, no antialiasing and fewer than 2^31 gaussians; anything else returns
 * GS_ERR_UNSUPPORTED (convert the features to f32 there).  Rows are padded to 8, 16, 40 or 64 channels (F <= 64) or to
 * 64-channel slices in the workspace; rows whose length is already that (F = 8, 16, 40, 64, 128, 192, 256) are read in
 * place and must be 16-byte aligned.  gs_raster_workspace_bytes sizes the bf16 layout (half the feature bytes). */

size_t gs_raster_workspace_bytes(const GsRasterParams* p);

/* gaussians2d (V,7) features (V,F) tile_ranges (T,2) int32 overlap_to_point (K) int32 ->
 * image (H,W,F) image_alpha (H,W) visibility (V; zeroed by the callee) or NULL */
int gs_raster_fwd(const GsRasterParams* p, const void* gaussians2d, const void* features,
                  const int32_t* tile_ranges, const int32_t* overlap_to_point, void* image,
                  void* image_alpha, void* visibility, void* workspace, size_t workspace_bytes,
                  void* stream);

/* image (H,W,F: forward output) grad_image (H,W,F) -> grad_gaussians (V,7) grad_features (V,F)
 * (each zeroed by the callee; NULL if the matching *_requires_grad is 0) and point_heuristic
 * (V,2), ACCUMULATED in place like backward.py:227-228 (the caller zero-fills it in forward).
 * Quantile mode (use_alpha_blending = 0; forward.py:107-114 has no backward in the reference): every pixel's image
 * gradient is added to the feature gradient of the gaussian the forward selected for it (the walk is replayed, `image`
 * may be NULL), grad_gaussians is zero (the selection is piecewise constant), point_heuristic is left untouched. */
int gs_raster_bwd(const GsRasterParams* p, const void* gaussians2d, const void* features,
                  const int32_t* tile_ranges, const int32_t* overlap_to_point, const void* image,
                  const void* grad_image, void* grad_gaussians, void* grad_features,
                  void* point_heuristic, void* workspace, size_t workspace_bytes, void* stream);

/* gs_raster_bwd with a differentiable image weight: image_weight (H,W: the forward's image_alpha) and its gradient
 * grad_image_weight (H,W).  The weight W = sum_i w_i is the blend of a constant feature 1, so its gradient flows into
 * grad_gaussians and point_heuristic exactly as that of one more channel of ones would (grad_features keeps F
 * columns).  grad_image_weight NULL: the same call as gs_raster_bwd, the same kernels.  Quantile mode
 * (use_alpha_blending = 0): the weight is W > 0, piecewise constant, and grad_image_weight is ignored.  With a weight
 * gradient the narrow backward (F <= 7) reduces every survivor alone (faster there than in pairs).
 * Extra cost per backward row: DESIGN.md §3. */
int gs_raster_bwd_with_weight(const GsRasterParams* p, const void* gaussians2d, const void* features,
                              const int32_t* tile_ranges, const int32_t* overlap_to_point, const void* image,
                              const void* grad_image, const void* image_weight, const void* grad_image_weight,
                              void* grad_gaussians, void* grad_features, void* point_heuristic, void* workspace,
                              size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ visibility-weighted sparse optimizers
 * (SURVEY.md 8f rank 1, the consumers of `visibility`): replace the per point step kernels of
 * optim/fractional_adam.py:7-85 and optim/fractional_laprop.py:7-86 together with the torch glue around them
 * (optim/fractional.py:108-151,186: local basis, mask_lr, point_lr, saturate, parameter update;
 * optim/visibility_aware.py:37-48,88-97: running visibility, weights, gradient rescaling).  f32 only, like the
 * reference's kernels.  `indexes` (M) int64 must be unique. */
typedef enum GsOptAlgorithm { GS_OPT_ADAM = 0, GS_OPT_LAPROP = 1 } GsOptAlgorithm;
typedef enum GsOptGroupType { GS_OPT_SCALAR = 0, GS_OPT_VECTOR = 1, GS_OPT_LOCAL_VECTOR = 2 } GsOptGroupType;

typedef struct GsOptParams {
  int32_t algorithm;       /* GsOptAlgorithm */
  int32_t group_type;      /* GsOptGroupType */
  int32_t dims;            /* D: columns of the parameter viewed as (N, D) */
  int32_t bias_correction;
  int64_t num_points;      /* N */
  int64_t num_visible;     /* M */
  double lr, beta1, beta2, eps;
  double grad_scale;       /* visibility-aware optimizers: grad * grad_scale / (visibility + vis_smooth) */
  double vis_smooth;       /* < 0: no visibility rescaling of the gradient (Fractional* / Sparse*) */
} GsOptParams;

/* running_vis (N), total_weight (N) updated in place; weight_out (M) = visibility / max(updated running vis, eps) */
int gs_opt_update_visibility(int64_t num_visible, const int64_t* indexes, const float* visibility,
                             float* running_vis, float* total_weight, float* weight_out, double vis_beta,
                             double eps, void* stream);
/* total_weight[indexes] += weight (Fractional* / Sparse*: optim/fractional.py:176) */
int gs_opt_accumulate_weight(int64_t num_visible, const int64_t* indexes, const float* weight,
                             float* total_weight, void* stream);
/* One fused update of a parameter group over the visible points.  grad, param (N, D); m (N, D); v (N, D) for scalar
 * groups, (N) for vector groups; total_weight (N) ALREADY updated for this step; weight (M); visibility (M) or NULL;
 * mask_lr (D) or NULL; point_lr (N) or NULL; basis (M, D, D) row major for local_vector groups (D = 2 or 3).
 * m, v and param are updated in place. */
int gs_opt_step(const GsOptParams* p, const int64_t* indexes, const float* weight, const float* visibility,
                const float* grad, float* m, float* v, const float* total_weight, float* param,
                const float* mask_lr, const float* point_lr, const float* basis, void* stream);

/* ------------------------------------------------------------------ Morton codes (SURVEY.md 8f rank 4)
 * replaces code_points32_kernel / code_points64_kernel (misc/morton_sort.py:93-111): the code of the grid cell
 * clamp((p - lower) / inc, 0, grid_size - 1) of every point, bits of x / y / z interleaved (x lowest).  points (n,3) f32;
 * lower, inc: 3 floats each ON THE DEVICE (so that the caller's min / resolution arithmetic needs no host sync);
 * code_bits 32 (grid_size <= 2^10, codes uint32) or 64 (grid_size <= 2^21, codes uint64).  Sorting the codes is
 * gs_radix_sort_pairs on 3 * log2(grid_size) bits. */
int gs_morton_codes(int64_t n, const float* points, const float* lower, const float* inc, int64_t grid_size,
                    int32_t code_bits, void* codes, void* stream);

/* ------------------------------------------------------------------ camera centre
 * replaces CameraParams.camera_position (perspective/params.py:75-78: torch.inverse(T_camera_world)[:3, 3], an LU
 * factorisation whose info check synchronises the host): position = -A^-1 t of the affine view matrix [A | t] held
 * row-major in T_camera_world (4x4, only the first three rows are read), A^-1 from cross products.  One thread, no
 * workspace, nothing read back.  dtype GS_F32 / GS_F64. */
int gs_camera_position(int32_t dtype, const void* T_camera_world, void* position, void* stream);

/* ------------------------------------------------------------------ multi-GPU: the step's gradient sum
 * The reference is single process (no collective call site); the view-parallel step of this package sums one flat f32
 * bucket over the ranks once per step (distributed.GradientBucket.all_reduce).  gs_multimem_all_reduce does that in
 * place through an NVSwitch MULTICAST mapping of the bucket (multicast_ptr: the address that stands for the same
 * offset on every GPU; the caller sets the mapping up — torch.distributed._symmetric_memory in this package): rank r
 * fetches the switch-reduced r-th slice with multimem.ld_reduce and writes it to all replicas with multimem.st.
 * flags_dev: DEVICE array of `world` pointers, entry q = rank q's flag words in peer-accessible memory,
 * gs_multimem_all_reduce_flag_words(world, num_blocks, num_channels) zero-initialised uint32 each; every rank must
 * launch with the same num_blocks (all of them resident: <= SMs of the device) and channel; reductions that can be in
 * flight at the same time use different channels.  Enqueued on `stream`; captured by CUDA graphs.
 * gs_cross_rank_barrier: the ranks meet on the stream (one CTA; the barrier of channel `channel` must not be shared
 * with a reduction in flight) — what every rank enqueued before it is complete and visible to its peers afterwards. */
int gs_multimem_all_reduce_flag_words(int32_t world, int32_t num_blocks, int32_t num_channels);
int gs_multimem_all_reduce(float* multicast_ptr, int64_t num_floats, int32_t rank, int32_t world,
                           uint32_t* const* flags_dev, int32_t num_blocks, int32_t channel, void* stream);
int gs_cross_rank_barrier(int32_t rank, int32_t world, uint32_t* const* flags_dev, int32_t num_blocks, int32_t channel,
                          void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GSPLAT_B200_H */
