// raster_fast_bwd_wide.cu — backward rasterizer for WIDE feature vectors (8..64 channels; f32, alpha blending,
// tile 16), e.g. BASELINE.json's feature-lifting configuration: depth + depth^2 + 32 features = 34 channels.
//
// Same arithmetic contract as raster_fast_bwd.cu (rasterizer/backward.py:52-228 of the reference).  With F
// channels the per pixel state of the narrow kernel (4 pixels per lane) no longer fits in registers, so the
// mapping is the forward kernel's: one CTA per 16x16 tile, 8 warps, a warp owns an 8x4 block, a lane ONE pixel.
//   * per pixel state in registers: W, RG = sum_c R_c G_c and the pixel's image gradient G[FP]; the replay needs
//     the remaining features only through R . G (see raster_fast_bwd.cu), so R itself is never materialised —
//     the reference keeps 2 x 4 x F floats per thread (backward.py:43-44,101-102);
//   * tile lists staged in batches of 32 through shared memory with cp.async double buffering (records + padded
//     feature rows, the 16 B chunks spread over the whole CTA); lane-parallel ellipse / block cull per warp;
//   * a lane is hit at most once per gaussian, so its feature-gradient contribution is just w G_c: the 7 (+2)
//     geometry sums and the F feature sums are reduced with transposed butterflies in groups of at most 32 values
//     (about one shuffle per value) and committed by the owning lanes with red.global.add.
// FP (padded channel count: 16, 36, 64) is a template parameter, F a runtime value; padded channels carry zeros.
#include "raster_fast.cuh"

namespace gs {

constexpr int kWideBatch = 32;
constexpr int kWideThreads = 256;

template <int FP, bool HEUR>
__global__ void __launch_bounds__(kWideThreads)
raster_bwd_wide_kernel(const __grid_constant__ GsRasterParams p, const float4* __restrict__ rec,
                       const float* __restrict__ featP, const int32_t* __restrict__ ranges,
                       const int32_t* __restrict__ o2p, const float* __restrict__ image,
                       const float* __restrict__ grad_image, float* __restrict__ grad_pts,
                       float* __restrict__ grad_feat, float* __restrict__ heuristic) {
  constexpr int NG = 7 + (HEUR ? 2 : 0);             // geometry (+ heuristic) values
  constexpr int C0 = FP < 32 ? FP : 32;              // first feature group
  constexpr int C1 = FP - C0;                        // second feature group (0, 4 or 32)
  __shared__ __align__(16) float4 s_r0[2][kWideBatch];
  __shared__ __align__(16) float4 s_r1[2][kWideBatch];
  __shared__ __align__(16) float s_feat[2][kWideBatch][FP];

  const int tile = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int tw = (p.image_width + kFastTile - 1) / kFastTile;
  const int F = p.num_features;
  const int wx0 = (tile % tw) * kFastTile + (warp & 1) * 8;
  const int wy0 = (tile / tw) * kFastTile + (warp >> 1) * 4;
  const int px = wx0 + (lane & 7), py = wy0 + (lane >> 3);
  const bool inb = px < p.image_width && py < p.image_height;
  const float pxf = (float)px + 0.5f, pyf = (float)py + 0.5f;
  const float bx0 = (float)wx0 + 0.5f, bx1 = (float)wx0 + 7.5f, by0 = (float)wy0 + 0.5f, by1 = (float)wy0 + 3.5f;
  const float thr = (float)p.alpha_threshold, cmax = (float)p.clamp_max_alpha, sat = (float)p.saturate_threshold;
  const float l2thr = log2f(thr);
  const bool pg = p.points_requires_grad && grad_pts != nullptr;
  const bool fg = p.features_requires_grad && grad_feat != nullptr;

  const int own_g = reduce_owner<NG>(lane);
  const int own_0 = reduce_owner<C0>(lane);
  const int own_1 = C1 > 0 ? reduce_owner<(C1 > 0 ? C1 : 1)>(lane) : -1;

  float G[FP];
  float W = inb ? 0.f : 1.f, RG = 0.f;
  {
    const int64_t pix = (int64_t)py * p.image_width + px;
#pragma unroll
    for (int c = 0; c < FP; ++c) {
      const bool ok = inb && c < F;
      G[c] = ok ? grad_image[pix * F + c] : 0.f;
      RG = fmaf(ok ? image[pix * F + c] : 0.f, G[c], RG);
    }
  }

  const int start = ranges[2 * tile], end = ranges[2 * tile + 1];
  const int C = end - start;
  const int nb = (C + kWideBatch - 1) / kWideBatch;

  auto issue_load = [&](int b) {
    const int buf = b & 1;
    if (t < kWideBatch) {
      const int v = b * kWideBatch + t;
      if (v < C) {
        const int idx = o2p[start + v];
        cp_async16(&s_r0[buf][t], rec + 2 * (int64_t)idx);
        cp_async16(&s_r1[buf][t], rec + 2 * (int64_t)idx + 1);
      }
    }
    constexpr int CH = FP / 4;
#pragma unroll
    for (int q0 = 0; q0 < kWideBatch * CH; q0 += kWideThreads) {
      const int q = q0 + t;
      const int slot = q / CH, part = q - slot * CH;
      const int v = b * kWideBatch + slot;
      if (q < kWideBatch * CH && v < C) {
        const int idx = o2p[start + v];
        cp_async16(&s_feat[buf][slot][part * 4], featP + (int64_t)idx * FP + part * 4);
      }
    }
    cp_async_commit();
  };

  bool warp_done = __all_sync(kFull, W >= sat);
  if (nb > 0) issue_load(0);
  for (int b = 0; b < nb; ++b) {
    const int buf = b & 1;
    if (b + 1 < nb) {
      issue_load(b + 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const int n_in = min(kWideBatch, C - b * kWideBatch);
    if (!warp_done) {
      bool touch = false;
      if (lane < n_in) {
        const float4 r0 = s_r0[buf][lane], r1 = s_r1[buf][lane];
        const float cx = kSqrtHalfLog2e * r1.x, cy = kSqrtHalfLog2e * r1.y;
        touch = block_may_touch(r0.x, r0.y, r0.z * cx, r0.w * cx, -r0.w * cy, r0.z * cy, log2f(r1.z) - l2thr, bx0, bx1,
                                by0, by1);
      }
      unsigned mask = __ballot_sync(kFull, touch);
      while (mask) {
        const int j = __ffs(mask) - 1;
        mask &= mask - 1;
        const float4 r0 = s_r0[buf][j], r1 = s_r1[buf][j];
        const float mx = r0.x, my = r0.y, ax = r0.z, ay = r0.w, isx = r1.x, isy = r1.y, a0 = r1.z;
        const float dx = pxf - mx, dy = pyf - my;
        const float tx = fmaf(dy, ay, dx * ax) * isx;
        const float ty = fmaf(dy, ax, -dx * ay) * isy;
        const float pgauss = fast_ex2(-kHalfLog2e * fmaf(ty, ty, tx * tx));
        float alpha = a0 * pgauss;
        const bool hit = alpha > thr && W < sat;
        if (!__any_sync(kFull, hit)) continue;

        float vg[NG];
#pragma unroll
        for (int k = 0; k < NG; ++k) vg[k] = 0.f;
        float wl = 0.f;  // this lane's blend weight for the gaussian (0 when not hit)
        if (hit) {
          alpha = fminf(alpha, cmax);
          const float Ti = 1.f - W;
          wl = alpha * Ti;
          W += wl;
          const float rinv = fast_rcp(1.f - alpha);
          float fG = 0.f;
#pragma unroll
          for (int c = 0; c < FP; c += 4) {
            const float4 f4 = *reinterpret_cast<const float4*>(&s_feat[buf][j][c]);
            fG = fmaf(f4.x, G[c], fG); fG = fmaf(f4.y, G[c + 1], fG);
            fG = fmaf(f4.z, G[c + 2], fG); fG = fmaf(f4.w, G[c + 3], fG);
          }
          RG = fmaf(-fG, wl, RG);
          const float ag = fmaf(fG, Ti, -RG * rinv);
          const float aag = a0 * ag;
          const float g = aag * pgauss;
          const float a = g * tx * isx, bq = g * ty * isy;
          vg[0] = fmaf(ax, a, -ay * bq); vg[1] = fmaf(ay, a, ax * bq);
          vg[2] = -fmaf(a, dx, bq * dy); vg[3] = fmaf(bq, dx, -a * dy);
          vg[4] = a * tx; vg[5] = bq * ty; vg[6] = pgauss * ag;
          if (HEUR) { vg[7] = aag * aag; vg[8] = fabsf(vg[0]) + fabsf(vg[1]); }
        }
        const int64_t idx = __float_as_int(r1.w);
        reduce_scatter_step<NG, 16>(vg, lane);
        if (own_g >= 0) {
          if (own_g < 7) { if (pg) atomicAdd(grad_pts + idx * 7 + own_g, vg[0]); }
          else if (HEUR) atomicAdd(heuristic + idx * 2 + (own_g - 7), vg[0]);
        }
        if (fg) {
          {
            float v[C0];
#pragma unroll
            for (int c = 0; c < C0; ++c) v[c] = wl * G[c];
            reduce_scatter_step<C0, 16>(v, lane);
            if (own_0 >= 0 && own_0 < F) atomicAdd(grad_feat + idx * F + own_0, v[0]);
          }
          if constexpr (C1 > 0) {
            float v[C1];
#pragma unroll
            for (int c = 0; c < C1; ++c) v[c] = wl * G[C0 + c];
            reduce_scatter_step<C1, 16>(v, lane);
            if (own_1 >= 0 && C0 + own_1 < F) atomicAdd(grad_feat + idx * F + C0 + own_1, v[0]);
          }
        }
      }
      warp_done = __all_sync(kFull, W >= sat);
    }
    if (__syncthreads_and(warp_done)) break;
  }
  cp_async_wait<0>();
}

// ------------------------------------------------------------------------------------------------ tensor-core variant
// With F channels the feature gradient of a gaussian over a warp's 8x4 pixel block is a vector-matrix product,
// d/df[c] = sum_p w[p] G[p][c]: the butterflies above spend ~4 instructions per channel and survivor on it (~150 of the
// ~300 instructions per survivor at F = 34).  Here a warp collects its survivors in groups of 16 and forms
//   D[16 survivors x F] = Wt[16 x 32 pixels] . G[32 pixels x F]
// on the tensor cores (mma.sync m16n8k8, tf32 inputs, f32 accumulate): the lanes park their blend weights in a
// per-warp shared-memory tile during the replay (one 8 B store per survivor), G sits in shared memory once per tile.
// tf32 alone (11 bit significands) would leave ~2e-4 relative error, above the 1e-4 gradient tolerance, so both
// operands are split x = hi + lo (both rounded to nearest tf32, residual 2^-24) and three products are accumulated
// (hi hi + lo hi + hi lo; the dropped lo lo term is 2^-22): measured error against the oracle as for the f32 path.
// Why mma.sync and not tcgen05: the product is per WARP (its own 16 survivors, its own 32 pixels), 16 x 32 x 40, issued
// from inside a SIMT replay loop whose A operand is produced by the lanes a few instructions earlier; a CTA-level
// tcgen05 tile (M >= 64, operands in descriptor-addressed shared memory, accumulator in TMEM behind an mbarrier) would
// need a block-diagonal [gaussians x 256 pixels] operand of mostly zeros and two extra copies for the split.  The tensor
// work is ~1 % of the kernel's issue slots either way; what it removes is the shuffle work.
constexpr int kMmaGroup = 16;   // survivors per product (M of the mma)
constexpr int kMmaBatch = 32;   // staged tile-list entries per buffer (64: 8.6 ms instead of 6.9 at config 4, the warps of a CTA drift further apart between barriers)

template <int FP>
struct WideMmaLayout {
  static constexpr int FP8 = (FP + 7) / 8 * 8;   // channels padded to n-tiles of 8
  static constexpr int NT = FP8 / 8;
  // row stride of the G tile (floats): = 8 or 24 mod 32 so that the B-fragment loads (row = lane & 3 (+4), column =
  // lane >> 2) hit 32 different banks
  static constexpr int GS = (FP8 % 32 == 8 || FP8 % 32 == 24) ? FP8 : FP8 + 8;
  static constexpr int WS = 36;                  // row stride of the weight tile (float2 units): conflict-free A loads
  static constexpr size_t stage_bytes = 2 * kMmaBatch * (32 + FP * 4);
  static constexpr size_t warp_bytes = 32 * GS * 4 + kMmaGroup * WS * 8 + kMmaGroup * 4;
  static constexpr size_t total(int warps) { return stage_bytes + warps * warp_bytes; }
};

// WARPS: warps per CTA = 8 (one CTA per tile) or 4 / 2 (two / four CTAs per tile, each staging the tile list for itself:
// the block barrier of a batch then waits for 4 / 2 warps instead of 8 — 21 % of the stall samples sat there).
// WGT: the image weight W is differentiable too (gradient gw, forward W in wimg): one more channel whose feature is
// always 1, so RG starts with W_final Gw and f . G gains + Gw (see raster_bwd_fast_kernel).
template <int FP, bool HEUR, int WARPS, bool WGT = false>
__global__ void __launch_bounds__(WARPS * 32, 16 / WARPS)   // 118 registers; an 80-register cap (three CTAs) spills: 8.0 vs 6.8 ms
raster_bwd_wide_mma_kernel(const __grid_constant__ GsRasterParams p, const float4* __restrict__ rec,
                           const float* __restrict__ featP, const int32_t* __restrict__ ranges,
                           const int32_t* __restrict__ o2p, const float* __restrict__ image,
                           const float* __restrict__ grad_image, float* __restrict__ grad_pts,
                           float* __restrict__ grad_feat, float* __restrict__ heuristic,
                           const float* __restrict__ wimg, const float* __restrict__ gw) {
  using L = WideMmaLayout<FP>;
  constexpr int NG = 7 + (HEUR ? 2 : 0);             // geometry (+ heuristic) values
  extern __shared__ __align__(16) unsigned char smem[];
  float4 (*s_r0)[kMmaBatch] = reinterpret_cast<float4 (*)[kMmaBatch]>(smem);
  float4 (*s_r1)[kMmaBatch] = reinterpret_cast<float4 (*)[kMmaBatch]>(smem + 2 * kMmaBatch * 16);
  float (*s_feat)[kMmaBatch][FP] = reinterpret_cast<float (*)[kMmaBatch][FP]>(smem + 2 * kMmaBatch * 32);

  constexpr int kThreads = WARPS * 32, kParts = 8 / WARPS;
  const int tile = blockIdx.x / kParts, t = threadIdx.x, lane = t & 31, lwarp = t >> 5;
  const int warp = (blockIdx.x % kParts) * WARPS + lwarp;   // which 8x4 pixel block of the tile
  unsigned char* wbase = smem + L::stage_bytes + (size_t)lwarp * L::warp_bytes;
  float* s_G = reinterpret_cast<float*>(wbase);                                    // [32][GS]
  float2* s_W = reinterpret_cast<float2*>(wbase + 32 * L::GS * 4);                 // [16][WS] {hi, lo}
  int* s_idx = reinterpret_cast<int*>(wbase + 32 * L::GS * 4 + kMmaGroup * L::WS * 8);   // [16]

  const int tw = (p.image_width + kFastTile - 1) / kFastTile;
  const int F = p.num_features;
  const int wx0 = (tile % tw) * kFastTile + (warp & 1) * 8;
  const int wy0 = (tile / tw) * kFastTile + (warp >> 1) * 4;
  const int px = wx0 + (lane & 7), py = wy0 + (lane >> 3);
  const bool inb = px < p.image_width && py < p.image_height;
  const float pxf = (float)px + 0.5f, pyf = (float)py + 0.5f;
  const float bx0 = (float)wx0 + 0.5f, bx1 = (float)wx0 + 7.5f, by0 = (float)wy0 + 0.5f, by1 = (float)wy0 + 3.5f;
  const float thr = (float)p.alpha_threshold, cmax = (float)p.clamp_max_alpha, sat = (float)p.saturate_threshold;
  const float l2thr = log2f(thr);
  const bool pg = p.points_requires_grad && grad_pts != nullptr;
  const bool fg = p.features_requires_grad && grad_feat != nullptr;
  const int own_g = reduce_owner<NG>(lane);
  const int gid = lane >> 2, tig = lane & 3;

  float G[FP];
  float W = inb ? 0.f : 1.f, RG = 0.f, Gw = 0.f;
  {
    const int64_t pix = (int64_t)py * p.image_width + px;
#pragma unroll
    for (int c = 0; c < FP; ++c) {
      const bool ok = inb && c < F;
      G[c] = ok ? grad_image[pix * F + c] : 0.f;
      RG = fmaf(ok ? image[pix * F + c] : 0.f, G[c], RG);
      s_G[lane * L::GS + c] = G[c];
    }
    if constexpr (WGT) {
      Gw = inb ? gw[pix] : 0.f;
      RG = fmaf(inb ? wimg[pix] : 0.f, Gw, RG);
    }
#pragma unroll
    for (int c = FP; c < L::FP8; ++c) s_G[lane * L::GS + c] = 0.f;
  }
  __syncwarp();

  int ns = 0;   // survivors parked in the weight tile (warp-uniform)

  // D = Wt . G for the parked survivors, committed with red.global.add (rows past ns hold stale weights: skipped)
  auto flush_group = [&]() {
    __syncwarp();
    if (fg) {
      unsigned ahi[4][4], alo[4][4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float2 a0 = s_W[gid * L::WS + tig + 8 * k], a1 = s_W[(gid + 8) * L::WS + tig + 8 * k];
        const float2 a2 = s_W[gid * L::WS + tig + 4 + 8 * k], a3 = s_W[(gid + 8) * L::WS + tig + 4 + 8 * k];
        ahi[k][0] = __float_as_uint(a0.x); ahi[k][1] = __float_as_uint(a1.x);
        ahi[k][2] = __float_as_uint(a2.x); ahi[k][3] = __float_as_uint(a3.x);
        alo[k][0] = __float_as_uint(a0.y); alo[k][1] = __float_as_uint(a1.y);
        alo[k][2] = __float_as_uint(a2.y); alo[k][3] = __float_as_uint(a3.y);
      }
      const int s0 = gid, s1 = gid + 8;
      const int64_t i0 = s0 < ns ? s_idx[s0] : -1, i1 = s1 < ns ? s_idx[s1] : -1;
#pragma unroll
      for (int n = 0; n < L::NT; ++n) {
        float c[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float b0 = s_G[(tig + 8 * k) * L::GS + gid + 8 * n], b1 = s_G[(tig + 4 + 8 * k) * L::GS + gid + 8 * n];
          const unsigned b0h = tf32_rna(b0), b1h = tf32_rna(b1);
          const unsigned b0l = tf32_rna(b0 - __uint_as_float(b0h)), b1l = tf32_rna(b1 - __uint_as_float(b1h));
          mma_tf32_16x8x8(c, ahi[k], b0h, b1h);
          mma_tf32_16x8x8(c, alo[k], b0h, b1h);
          mma_tf32_16x8x8(c, ahi[k], b0l, b1l);
        }
        const int ch = 8 * n + 2 * tig;
        if (i0 >= 0) {
          if (ch < F) atomicAdd(grad_feat + i0 * F + ch, c[0]);
          if (ch + 1 < F) atomicAdd(grad_feat + i0 * F + ch + 1, c[1]);
        }
        if (i1 >= 0) {
          if (ch < F) atomicAdd(grad_feat + i1 * F + ch, c[2]);
          if (ch + 1 < F) atomicAdd(grad_feat + i1 * F + ch + 1, c[3]);
        }
      }
    }
    ns = 0;
    __syncwarp();   // the tile is free for the next group's stores
  };

  const int start = ranges[2 * tile], end = ranges[2 * tile + 1];
  const int C = end - start;
  const int nb = (C + kMmaBatch - 1) / kMmaBatch;

  auto issue_load = [&](int b) {
    const int buf = b & 1;
    if (t < kMmaBatch) {
      const int v = b * kMmaBatch + t;
      if (v < C) {
        const int idx = o2p[start + v];
        cp_async16(&s_r0[buf][t], rec + 2 * (int64_t)idx);
        cp_async16(&s_r1[buf][t], rec + 2 * (int64_t)idx + 1);
      }
    }
    constexpr int CH = FP / 4;
#pragma unroll
    for (int q0 = 0; q0 < kMmaBatch * CH; q0 += kThreads) {
      const int q = q0 + t;
      const int slot = q / CH, part = q - slot * CH;
      const int v = b * kMmaBatch + slot;
      if (q < kMmaBatch * CH && v < C) {
        const int idx = o2p[start + v];
        cp_async16(&s_feat[buf][slot][part * 4], featP + (int64_t)idx * FP + part * 4);
      }
    }
    cp_async_commit();
  };

  bool warp_done = __all_sync(kFull, W >= sat);
  if (nb > 0) issue_load(0);
  for (int b = 0; b < nb; ++b) {
    const int buf = b & 1;
    if (b + 1 < nb) {
      issue_load(b + 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const int n_in = min(kMmaBatch, C - b * kMmaBatch);
    if (!warp_done) {
     for (int c0 = 0; c0 < n_in; c0 += 32) {
      bool touch = false;
      if (c0 + lane < n_in) {
        const float4 r0 = s_r0[buf][c0 + lane], r1 = s_r1[buf][c0 + lane];
        const float cx = kSqrtHalfLog2e * r1.x, cy = kSqrtHalfLog2e * r1.y;
        touch = block_may_touch(r0.x, r0.y, r0.z * cx, r0.w * cx, -r0.w * cy, r0.z * cy, log2f(r1.z) - l2thr, bx0, bx1,
                                by0, by1);
      }
      unsigned mask = __ballot_sync(kFull, touch);
      while (mask) {
        const int j = c0 + __ffs(mask) - 1;
        mask &= mask - 1;
        const float4 r0 = s_r0[buf][j], r1 = s_r1[buf][j];
        const float mx = r0.x, my = r0.y, ax = r0.z, ay = r0.w, isx = r1.x, isy = r1.y, a0 = r1.z;
        const float dx = pxf - mx, dy = pyf - my;
        const float tx = fmaf(dy, ay, dx * ax) * isx;
        const float ty = fmaf(dy, ax, -dx * ay) * isy;
        const float pgauss = fast_ex2(-kHalfLog2e * fmaf(ty, ty, tx * tx));
        float alpha = a0 * pgauss;
        const bool hit = alpha > thr && W < sat;
        if (!__any_sync(kFull, hit)) continue;

        float vg[NG];
#pragma unroll
        for (int k = 0; k < NG; ++k) vg[k] = 0.f;
        float wl = 0.f;  // this lane's blend weight for the gaussian (0 when not hit)
        if (hit) {
          alpha = fminf(alpha, cmax);
          const float Ti = 1.f - W;
          wl = alpha * Ti;
          W += wl;
          const float rinv = fast_rcp(1.f - alpha);
          float fG0 = 0.f, fG1 = 0.f, fG2 = 0.f, fG3 = 0.f;   // four independent chains: the dot product is latency bound
#pragma unroll
          for (int c = 0; c < FP; c += 4) {
            const float4 f4 = *reinterpret_cast<const float4*>(&s_feat[buf][j][c]);
            fG0 = fmaf(f4.x, G[c], fG0); fG1 = fmaf(f4.y, G[c + 1], fG1);
            fG2 = fmaf(f4.z, G[c + 2], fG2); fG3 = fmaf(f4.w, G[c + 3], fG3);
          }
          float fG = (fG0 + fG1) + (fG2 + fG3);
          if constexpr (WGT) fG += Gw;
          RG = fmaf(-fG, wl, RG);
          const float ag = fmaf(fG, Ti, -RG * rinv);
          const float aag = a0 * ag;
          const float g = aag * pgauss;
          const float a = g * tx * isx, bq = g * ty * isy;
          vg[0] = fmaf(ax, a, -ay * bq); vg[1] = fmaf(ay, a, ax * bq);
          vg[2] = -fmaf(a, dx, bq * dy); vg[3] = fmaf(bq, dx, -a * dy);
          vg[4] = a * tx; vg[5] = bq * ty; vg[6] = pgauss * ag;
          if (HEUR) { vg[7] = aag * aag; vg[8] = fabsf(vg[0]) + fabsf(vg[1]); }
        }
        const int64_t idx = __float_as_int(r1.w);
        reduce_scatter_step<NG, 16>(vg, lane);
        if (own_g >= 0) {
          if (own_g < 7) { if (pg) atomicAdd(grad_pts + idx * 7 + own_g, vg[0]); }
          else if (HEUR) atomicAdd(heuristic + idx * 2 + (own_g - 7), vg[0]);
        }
        if (fg) {   // park the blend weights of this survivor: row ns of the warp's weight tile
          const float whi = __uint_as_float(tf32_rna(wl));
          s_W[ns * L::WS + lane] = make_float2(whi, __uint_as_float(tf32_rna(wl - whi)));
          if (lane == 0) s_idx[ns] = (int)idx;
          if (++ns == kMmaGroup) flush_group();
        }
      }
     }
      warp_done = __all_sync(kFull, W >= sat);
    }
    if (__syncthreads_and(warp_done)) break;
  }
  cp_async_wait<0>();
  if (ns > 0) flush_group();
}

template <int FP, bool HEUR, int WARPS, bool WGT = false>
static int launch_wide_mma_w(const GsRasterParams& p, const RasterArgs& a, const float4* rec, const float* featP, int tiles,
                             cudaStream_t st) {
  using L = WideMmaLayout<FP>;
  // per launch: the attribute belongs to the (function, device) pair and the call costs about a microsecond
  GS_CUDA(cudaFuncSetAttribute(raster_bwd_wide_mma_kernel<FP, HEUR, WARPS, WGT>,
                               cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L::total(WARPS)));
  raster_bwd_wide_mma_kernel<FP, HEUR, WARPS, WGT><<<tiles * (8 / WARPS), WARPS * 32, L::total(WARPS), st>>>(
      p, rec, featP, a.tile_ranges, a.overlap_to_point, (const float*)a.image_in, (const float*)a.grad_image,
      (float*)a.grad_gaussians, (float*)a.grad_features, HEUR ? (float*)a.point_heuristic : nullptr,
      (const float*)a.image_weight, (const float*)a.grad_image_weight);
  return GS_OK;
}

template <int FP, bool HEUR>
static int launch_wide_mma(const GsRasterParams& p, const RasterArgs& a, const float4* rec, const float* featP, int tiles,
                           cudaStream_t st) {
  // Two warps per CTA (four CTAs per tile).  Measured at config 4 (34 channels, 4K; benchmarks/variants.py
  // --variants 0,8,16,24 --scene c4): eight warps 7.05 ms, four 7.35, two 6.39, one 6.99.
  // kernel_variant bits 3-4 (A/B): 0 = two warps per CTA, 1 = eight, 2 = four, 3 = one.  With the weight gradient
  // only the shipped two-warp kernel exists.
  if (a.grad_image_weight != nullptr) return launch_wide_mma_w<FP, HEUR, 2, true>(p, a, rec, featP, tiles, st);
  switch ((p.kernel_variant >> 3) & 3) {
    case 1: return launch_wide_mma_w<FP, HEUR, 8>(p, a, rec, featP, tiles, st);
    case 2: return launch_wide_mma_w<FP, HEUR, 4>(p, a, rec, featP, tiles, st);
    case 3: return launch_wide_mma_w<FP, HEUR, 1>(p, a, rec, featP, tiles, st);
    default: return launch_wide_mma_w<FP, HEUR, 2>(p, a, rec, featP, tiles, st);
  }
}

int raster_bwd_wide(const GsRasterParams& p, const RasterArgs& a, const float4* rec, const float* featP,
                    cudaStream_t st) {
  const int tiles = tiles_wide(p) * tiles_high(p);
  const bool heur = p.compute_point_heuristic && a.point_heuristic != nullptr;
  // tensor-core feature gradient (kernel_variant bit 1 = the butterfly kernel, which has no weight gradient)
  if ((p.kernel_variant & 2) == 0 || a.grad_image_weight != nullptr) {
    int rc = GS_OK;
#define GS_WIDE_MMA_CASE(FPV) \
  case FPV: rc = heur ? launch_wide_mma<FPV, true>(p, a, rec, featP, tiles, st) \
                      : launch_wide_mma<FPV, false>(p, a, rec, featP, tiles, st); break
    switch (fast_feature_pad(p.num_features)) {
      GS_WIDE_MMA_CASE(8);
      GS_WIDE_MMA_CASE(16);
      GS_WIDE_MMA_CASE(36);
      GS_WIDE_MMA_CASE(64);
      default: GS_UNSUPPORTED("rasterizer backward (wide): %d feature channels", p.num_features);
    }
#undef GS_WIDE_MMA_CASE
    if (rc != GS_OK) return rc;
    GS_LAUNCH_CHECK();
    return GS_OK;
  }
#define GS_WIDE_LAUNCH(FPV, HEURV)                                                                                  \
  raster_bwd_wide_kernel<FPV, HEURV><<<tiles, kWideThreads, 0, st>>>(                                              \
      p, rec, featP, a.tile_ranges, a.overlap_to_point, (const float*)a.image_in, (const float*)a.grad_image,      \
      (float*)a.grad_gaussians, (float*)a.grad_features, heur ? (float*)a.point_heuristic : nullptr)
#define GS_WIDE_CASE(FPV) \
  case FPV: if (heur) GS_WIDE_LAUNCH(FPV, true); else GS_WIDE_LAUNCH(FPV, false); break
  switch (fast_feature_pad(p.num_features)) {
    GS_WIDE_CASE(8);
    GS_WIDE_CASE(16);
    GS_WIDE_CASE(36);
    GS_WIDE_CASE(64);
    default: GS_UNSUPPORTED("rasterizer backward (wide): %d feature channels", p.num_features);
  }
#undef GS_WIDE_CASE
#undef GS_WIDE_LAUNCH
  GS_LAUNCH_CHECK();
  return GS_OK;
}

}  // namespace gs
