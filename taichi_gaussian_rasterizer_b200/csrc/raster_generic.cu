// raster_generic.cu — the general rasterizer kernels: any dtype (f32 / f64), tile size 8 / 16 / 32,
// antialiased or plain gaussian evaluation, alpha blending or quantile mode, visibility, heuristics.
// One CTA per tile, one pixel per thread, the tile's depth-sorted gaussians staged through shared
// memory in groups of tile_size^2 exactly as the reference does — including its literal group-size
// arithmetic (forward.py:88) when p.emulate_stale_tail is set, so the "stale tail" (SURVEY Q1) arises
// from the same structure.  The f32 / blending / tile-16 case normally takes the faster kernels in
// raster_fast_*.cu; this file is the fidelity-first path and the f64 gradcheck path.
//
// Replaces rasterizer/forward.py:24-137 and rasterizer/backward.py:52-228 of
// /root/reference/taichi_splatting/.
#include "raster.cuh"
#include "raster_math.cuh"

namespace gs {

// MODE kBlend: alpha blending.  kQuantile: the feature of the gaussian at which the accumulated weight first reaches
// 1 - saturate_threshold (forward.py:107-114).  kQuantileBwd: the same walk, but instead of writing the image each
// pixel adds its image gradient to the feature gradient of the gaussian it selected — the backward of quantile mode
// (SURVEY 8f rank 3; the reference has none, tests/test_rasterizer.py:92-94).  The selection is piecewise constant in
// the gaussians' geometry and opacity, so their gradient is zero almost everywhere and is returned as zeros.
constexpr int kBlend = 1, kQuantile = 0, kQuantileBwd = 2;

template <typename T, int MAXF, bool AA, int MODE, int NT>
__global__ void __launch_bounds__(NT) raster_fwd_generic_kernel(const __grid_constant__ GsRasterParams p, const T* __restrict__ pts,
                                          const T* __restrict__ feat, const int32_t* __restrict__ ranges,
                                          const int32_t* __restrict__ o2p, T* __restrict__ image,
                                          T* __restrict__ image_alpha, T* __restrict__ visibility,
                                          const T* __restrict__ grad_image, T* __restrict__ grad_feat) {
  constexpr bool BLEND = MODE == kBlend;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int ts = p.tile_size, A = ts * ts, F = p.num_features;
  T* s_pts = reinterpret_cast<T*>(smem_raw);
  T* s_feat = s_pts + A * 7;
  T* s_vis = s_feat + A * F;
  int* s_id = reinterpret_cast<int*>(s_vis + A);

  const int tile = blockIdx.x, t = threadIdx.x, lane = t & 31;
  const int tw = (p.image_width + ts - 1) / ts;
  const int px = (tile % tw) * ts + t % ts, py = (tile / tw) * ts + t / ts;
  const bool inb = px < p.image_width && py < p.image_height;
  const T pxf = T(px) + T(0.5), pyf = T(py) + T(0.5);
  const T thr = T(p.alpha_threshold), cmax = T(p.clamp_max_alpha);
  const T sat_w = T(1.0 - p.saturate_threshold), exit_T = T(p.forward_exit_transmittance);
  const bool want_vis = MODE != kQuantileBwd && p.compute_visibility && visibility != nullptr;

  T acc[MAXF];  // kQuantileBwd: the pixel's image gradient
#pragma unroll
  for (int c = 0; c < MAXF; ++c) acc[c] = T(0);
  if (MODE == kQuantileBwd && inb) {
#pragma unroll
    for (int c = 0; c < MAXF; ++c)
      if (c < F) acc[c] = grad_image[((int64_t)py * p.image_width + px) * F + c];
  }
  T W = inb ? T(0) : T(1);
  bool saturated = false;
  bool done = BLEND ? ((T(1) - W) <= exit_T) : false;

  const int start = ranges[2 * tile], end = ranges[2 * tile + 1];
  const int C = end - start;
  const int G = (C + A - 1) / A;
  for (int grp = 0; grp < G; ++grp) {
    if (__syncthreads_and(done || !inb)) break;
    const int load_index = start + grp * A + t;
    if (load_index < end) {
      const int idx = o2p[load_index];
#pragma unroll
      for (int k = 0; k < 7; ++k) s_pts[t * 7 + k] = pts[(int64_t)idx * 7 + k];
      if (MODE != kQuantileBwd)
        for (int c = 0; c < F; ++c) s_feat[t * F + c] = feat[(int64_t)idx * F + c];
      s_id[t] = idx;
      s_vis[t] = T(0);
    }
    __syncthreads();
    const int remaining = p.emulate_stale_tail ? (C - grp) : (C - grp * A);
    const int iters = remaining < A ? remaining : A;
    for (int s = 0; s < iters; ++s) {
      if (__all_sync(kFull, done || !inb)) break;
      T weight = T(0);
      if (!done && inb) {
        const Gauss2D<T> g = load_gauss<T>(s_pts + s * 7);
        const T ga = AA ? pdf_aa<T>(pxf, pyf, g) : pdf<T>(pxf, pyf, g);
        T alpha = g.alpha * ga;
        alpha = alpha < cmax ? alpha : cmax;
        if (alpha > thr) {
          weight = alpha * (T(1) - W);
          W += weight;
          if (BLEND) {
#pragma unroll
            for (int c = 0; c < MAXF; ++c)
              if (c < F) acc[c] += s_feat[s * F + c] * weight;
          } else {
            if (W >= sat_w && !saturated) {
#pragma unroll
              for (int c = 0; c < MAXF; ++c) {
                if (c < F) {
                  if (MODE == kQuantileBwd) red_add(grad_feat + (int64_t)s_id[s] * F + c, acc[c]);
                  else acc[c] = s_feat[s * F + c];
                }
              }
            }
            saturated = W >= sat_w;
          }
        }
        done = BLEND ? ((T(1) - W) <= exit_T) : saturated;
      }
      if (want_vis) {
        if (__any_sync(kFull, weight > T(0))) {
          const T v = warp_sum(weight);
          if (lane == 0) atomicAdd(&s_vis[s], v);
        }
      }
    }
    if (want_vis) {
      __syncthreads();
      if (load_index < end) red_add(visibility + s_id[t], s_vis[t]);
    }
  }
  if (MODE != kQuantileBwd && inb) {
    const int64_t pix = (int64_t)py * p.image_width + px;
#pragma unroll
    for (int c = 0; c < MAXF; ++c)
      if (c < F) image[pix * F + c] = acc[c];
    image_alpha[pix] = BLEND ? W : T(W > T(0));
  }
}

// WGT: the image weight W = sum_i w_i is differentiable too (gradient gw, forward W in wimg).  W is the blend of a
// constant feature 1: its remaining part Rw starts at W_final, Rw -= w per hit, and dL/dalpha gains (T - Rw / (1 - alpha)) Gw.
template <typename T, int MAXF, bool AA, int NT, bool WGT = false>
__global__ void __launch_bounds__(NT) raster_bwd_generic_kernel(const __grid_constant__ GsRasterParams p, int batch,
                                          const T* __restrict__ pts, const T* __restrict__ feat,
                                          const int32_t* __restrict__ ranges, const int32_t* __restrict__ o2p,
                                          const T* __restrict__ image, const T* __restrict__ grad_image,
                                          T* __restrict__ grad_pts, T* __restrict__ grad_feat,
                                          T* __restrict__ heuristic, const T* __restrict__ wimg,
                                          const T* __restrict__ gw) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int ts = p.tile_size, F = p.num_features, B = batch;
  T* s_pts = reinterpret_cast<T*>(smem_raw);  // B*7
  T* s_feat = s_pts + B * 7;                  // B*F
  T* s_gp = s_feat + B * F;                   // B*7
  T* s_gf = s_gp + B * 7;                     // B*F
  T* s_h = s_gf + B * F;                      // B*2
  int* s_id = reinterpret_cast<int*>(s_h + B * 2);

  const int tile = blockIdx.x, t = threadIdx.x, lane = t & 31;
  const int tw = (p.image_width + ts - 1) / ts;
  const int px = (tile % tw) * ts + t % ts, py = (tile / tw) * ts + t / ts;
  const bool inb = px < p.image_width && py < p.image_height;
  const T pxf = T(px) + T(0.5), pyf = T(py) + T(0.5);
  const T thr = T(p.alpha_threshold), cmax = T(p.clamp_max_alpha), sat = T(p.saturate_threshold);
  const bool pg = p.points_requires_grad && grad_pts != nullptr;
  const bool fg = p.features_requires_grad && grad_feat != nullptr;
  const bool hg = p.compute_point_heuristic && heuristic != nullptr;

  T R[MAXF], Gp[MAXF];
  T W = T(1), Rw = T(0), Gw = T(0);
#pragma unroll
  for (int c = 0; c < MAXF; ++c) { R[c] = T(0); Gp[c] = T(0); }
  if (inb) {
    const int64_t pix = (int64_t)py * p.image_width + px;
#pragma unroll
    for (int c = 0; c < MAXF; ++c)
      if (c < F) { R[c] = image[pix * F + c]; Gp[c] = grad_image[pix * F + c]; }
    if constexpr (WGT) { Rw = wimg[pix]; Gw = gw[pix]; }
    W = T(0);
  }

  const int start = ranges[2 * tile], end = ranges[2 * tile + 1];
  const int C = end - start;
  const int G = (C + B - 1) / B;
  for (int grp = 0; grp < G; ++grp) {
    if (__syncthreads_and(W >= sat)) break;
    const int gstart = start + grp * B;
    const int n_in = (end - gstart) < B ? (end - gstart) : B;
    if (t < n_in) {
      const int idx = o2p[gstart + t];
#pragma unroll
      for (int k = 0; k < 7; ++k) { s_pts[t * 7 + k] = pts[(int64_t)idx * 7 + k]; s_gp[t * 7 + k] = T(0); }
      for (int c = 0; c < F; ++c) { s_feat[t * F + c] = feat[(int64_t)idx * F + c]; s_gf[t * F + c] = T(0); }
      s_h[t * 2] = T(0); s_h[t * 2 + 1] = T(0);
      s_id[t] = idx;
    }
    __syncthreads();
    for (int s = 0; s < n_in; ++s) {
      if (__all_sync(kFull, W >= sat)) break;
      T gp[7] = {T(0), T(0), T(0), T(0), T(0), T(0), T(0)};
      T gf[MAXF];
#pragma unroll
      for (int c = 0; c < MAXF; ++c) gf[c] = T(0);
      T h0 = T(0), h1 = T(0);
      bool has_grad = false;
      const Gauss2D<T> g = load_gauss<T>(s_pts + s * 7);
      const PdfGrad<T> d = AA ? pdf_aa_grad<T>(pxf, pyf, g) : pdf_grad<T>(pxf, pyf, g);
      T alpha = g.alpha * d.p;
      if (alpha > thr && !(W >= sat)) {
        has_grad = true;
        alpha = alpha < cmax ? alpha : cmax;
        const T Ti = T(1) - W;
        const T weight = alpha * Ti;
        W += weight;
        T alpha_grad = T(0);
#pragma unroll
        for (int c = 0; c < MAXF; ++c)
          if (c < F) {
            const T f = s_feat[s * F + c];
            R[c] -= f * weight;
            const T diff = f * Ti - R[c] / (T(1) - alpha);
            alpha_grad += diff * Gp[c];
            gf[c] = weight * Gp[c];
          }
        if constexpr (WGT) {
          Rw -= weight;
          alpha_grad += (Ti - Rw / (T(1) - alpha)) * Gw;
        }
        const T aag = g.alpha * alpha_grad;
        gp[0] = aag * d.dmx; gp[1] = aag * d.dmy;
        gp[2] = aag * d.dax; gp[3] = aag * d.day;
        gp[4] = aag * d.dsx; gp[5] = aag * d.dsy;
        gp[6] = d.p * alpha_grad;
        h0 = aag * aag;
        h1 = fabs(gp[0]) + fabs(gp[1]);
      }
      if (__any_sync(kFull, has_grad)) {
        if (pg) {
#pragma unroll
          for (int k = 0; k < 7; ++k) {
            const T v = warp_sum(gp[k]);
            if (lane == 0) atomicAdd(&s_gp[s * 7 + k], v);
          }
        }
        if (fg) {
#pragma unroll
          for (int c = 0; c < MAXF; ++c)
            if (c < F) {
              const T v = warp_sum(gf[c]);
              if (lane == 0) atomicAdd(&s_gf[s * F + c], v);
            }
        }
        if (hg) {
          const T v0 = warp_sum(h0), v1 = warp_sum(h1);
          if (lane == 0) { atomicAdd(&s_h[s * 2], v0); atomicAdd(&s_h[s * 2 + 1], v1); }
        }
      }
    }
    __syncthreads();
    if (t < n_in) {
      const int64_t idx = s_id[t];
      if (pg) {
#pragma unroll
        for (int k = 0; k < 7; ++k) red_add(grad_pts + idx * 7 + k, s_gp[t * 7 + k]);
      }
      if (fg)
        for (int c = 0; c < F; ++c) red_add(grad_feat + idx * F + c, s_gf[t * F + c]);
      if (hg) { red_add(heuristic + idx * 2, s_h[t * 2]); red_add(heuristic + idx * 2 + 1, s_h[t * 2 + 1]); }
    }
  }
}

template <typename T, int MAXF, bool AA, int MODE, int NT>
static int launch_fwd(const GsRasterParams& p, const RasterArgs& a, cudaStream_t st) {
  const int A = p.tile_size * p.tile_size;
  const size_t smem = (size_t)A * (7 + p.num_features + 1) * sizeof(T) + (size_t)A * sizeof(int);
  auto kern = raster_fwd_generic_kernel<T, MAXF, AA, MODE, NT>;
  if (smem > 48 * 1024) GS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int tiles = tiles_wide(p) * tiles_high(p);
  kern<<<tiles, A, smem, st>>>(p, (const T*)a.gaussians2d, (const T*)a.features, a.tile_ranges, a.overlap_to_point,
                               (T*)a.image, (T*)a.image_alpha, (T*)a.visibility, (const T*)a.grad_image,
                               (T*)a.grad_features);
  GS_LAUNCH_CHECK();
  return GS_OK;
}

template <typename T, int MAXF, bool AA, int NT, bool WGT>
static int launch_bwd(const GsRasterParams& p, const RasterArgs& a, cudaStream_t st) {
  const int A = p.tile_size * p.tile_size;
  const int B = A < 256 ? A : 256;
  const size_t smem = (size_t)B * ((7 + p.num_features) * 2 + 2) * sizeof(T) + (size_t)B * sizeof(int);
  auto kern = raster_bwd_generic_kernel<T, MAXF, AA, NT, WGT>;
  if (smem > 48 * 1024) GS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int tiles = tiles_wide(p) * tiles_high(p);
  kern<<<tiles, A, smem, st>>>(p, B, (const T*)a.gaussians2d, (const T*)a.features, a.tile_ranges, a.overlap_to_point,
                               (const T*)a.image_in, (const T*)a.grad_image, (T*)a.grad_gaussians,
                               (T*)a.grad_features, (T*)a.point_heuristic, (const T*)a.image_weight,
                               (const T*)a.grad_image_weight);
  GS_LAUNCH_CHECK();
  return GS_OK;
}

template <typename T, int MAXF, int NT>
static int fwd_modes(const GsRasterParams& p, const RasterArgs& a, cudaStream_t st) {
  if (p.antialias) return p.use_alpha_blending ? launch_fwd<T, MAXF, true, kBlend, NT>(p, a, st)
                                               : launch_fwd<T, MAXF, true, kQuantile, NT>(p, a, st);
  return p.use_alpha_blending ? launch_fwd<T, MAXF, false, kBlend, NT>(p, a, st)
                              : launch_fwd<T, MAXF, false, kQuantile, NT>(p, a, st);
}

template <typename T, int MAXF, int NT>
static int bwd_modes(const GsRasterParams& p, const RasterArgs& a, cudaStream_t st) {
  if (!p.use_alpha_blending) {  // quantile mode: replay the forward's selection, scatter the image gradient
    if (!p.features_requires_grad || a.grad_features == nullptr) return GS_OK;
    return p.antialias ? launch_fwd<T, MAXF, true, kQuantileBwd, NT>(p, a, st)
                       : launch_fwd<T, MAXF, false, kQuantileBwd, NT>(p, a, st);
  }
  if (a.grad_image_weight != nullptr)
    return p.antialias ? launch_bwd<T, MAXF, true, NT, true>(p, a, st) : launch_bwd<T, MAXF, false, NT, true>(p, a, st);
  return p.antialias ? launch_bwd<T, MAXF, true, NT, false>(p, a, st) : launch_bwd<T, MAXF, false, NT, false>(p, a, st);
}

int raster_fwd_generic(const GsRasterParams& p, const RasterArgs& a, cudaStream_t st) {
  const int F = p.num_features;
  const bool big = p.tile_size == 32;  // 1024 threads per CTA: register budget 64, small feature counts only
  if (p.dtype == GS_F32) {
    if (big) {
      if (F <= 4) return fwd_modes<float, 4, 1024>(p, a, st);
      if (F <= 8) return fwd_modes<float, 8, 1024>(p, a, st);
      GS_UNSUPPORTED("rasterizer forward: tile_size 32 supports up to 8 feature channels, got %d", F);
    }
    if (F <= 4) return fwd_modes<float, 4, 256>(p, a, st);
    if (F <= 8) return fwd_modes<float, 8, 256>(p, a, st);
    if (F <= 16) return fwd_modes<float, 16, 256>(p, a, st);
    if (F <= 40) return fwd_modes<float, 40, 256>(p, a, st);
    GS_UNSUPPORTED("rasterizer forward: %d feature channels (f32 supports up to 40, or up to 256 with "
                   "tile_size 16, alpha blending and no antialiasing)", F);
  }
  if (big) {
    if (F <= 4) return fwd_modes<double, 4, 1024>(p, a, st);
    GS_UNSUPPORTED("rasterizer forward: f64 tile_size 32 supports up to 4 feature channels, got %d", F);
  }
  if (F <= 4) return fwd_modes<double, 4, 256>(p, a, st);
  if (F <= 8) return fwd_modes<double, 8, 256>(p, a, st);
  GS_UNSUPPORTED("rasterizer forward: %d feature channels (f64 supports up to 8)", F);
}

int raster_bwd_generic(const GsRasterParams& p, const RasterArgs& a, cudaStream_t st) {
  const int F = p.num_features;
  const bool big = p.tile_size == 32;
  if (p.dtype == GS_F32) {
    if (big) {
      if (F <= 4) return bwd_modes<float, 4, 1024>(p, a, st);
      if (F <= 8) return bwd_modes<float, 8, 1024>(p, a, st);
      GS_UNSUPPORTED("rasterizer backward: tile_size 32 supports up to 8 feature channels, got %d", F);
    }
    if (F <= 4) return bwd_modes<float, 4, 256>(p, a, st);
    if (F <= 8) return bwd_modes<float, 8, 256>(p, a, st);
    if (F <= 16) return bwd_modes<float, 16, 256>(p, a, st);
    if (F <= 40) return bwd_modes<float, 40, 256>(p, a, st);
    GS_UNSUPPORTED("rasterizer backward: %d feature channels (f32 supports up to 40, or up to 256 with "
                   "tile_size 16, alpha blending and no antialiasing)", F);
  }
  if (big) {
    if (F <= 4) return bwd_modes<double, 4, 1024>(p, a, st);
    GS_UNSUPPORTED("rasterizer backward: f64 tile_size 32 supports up to 4 feature channels, got %d", F);
  }
  if (F <= 4) return bwd_modes<double, 4, 256>(p, a, st);
  if (F <= 8) return bwd_modes<double, 8, 256>(p, a, st);
  GS_UNSUPPORTED("rasterizer backward: %d feature channels (f64 supports up to 8)", F);
}

}  // namespace gs
