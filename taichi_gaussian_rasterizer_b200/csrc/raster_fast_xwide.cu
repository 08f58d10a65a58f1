// raster_fast_xwide.cu — backward rasterizer for EXTRA-WIDE feature vectors (65..256 channels; f32, alpha blending,
// tile 16): feature fields for semantic or foundation-model distillation (128, 256 dimensions) in one pass.
//
// The forward is raster_fwd_fast_kernel<64, ..., XW = true> (raster_fast_fwd.cu): one CTA per tile and 64-channel
// slice.  The backward cannot be sliced that way: aag = alpha_0 * alpha_grad enters the heuristics as aag^2 and
// |pgx| + |pgy|, which are not linear in the channels, and alpha_grad itself needs the full dot product G . f_i.
// So this kernel keeps the mapping of raster_bwd_wide_mma_kernel (raster_fast_bwd_wide.cu): a warp owns an 8x4 pixel
// block, a lane ONE pixel; the replay uses the R . G identity
//     alpha_grad = T (G . f_i) - RG / (1 - alpha),   RG -= w (G . f_i)
// and the feature gradient sum_px w G of a group of 16 survivors is a [16 survivors x 32 pixels] . [32 pixels x F]
// product on the tensor cores, split tf32 (hi / lo, three products: the same accuracy as the wide kernel).
// What changes with F:
//   * the pixel's image gradient G (up to 256 floats) no longer fits in registers: it sits in the warp's shared-memory
//     tile [32 pixels][FP + 4], read by the dot product (a lane reads its own row with LDS.128: the row stride, 4 mod
//     32 banks, keeps those conflict free) and by the product's B fragments (two-way bank conflicts there);
//   * tile lists are staged in batches of 16 entries (records + full feature rows) so that at F = 256 two CTAs of two
//     warps fit an SM (2 x 107 KB of shared memory); 32 px x 256 ch x 4 B = 32 KB of G per warp is what limits that.
// Why G . f_i stays on the SIMT pipes: it is needed only for the lanes a survivor hits, inside the sequential replay,
// and costs F / 4 LDS.128 + F FFMA per hit lane; as a [candidates x F] . [F x 32 pixels] product it would be formed
// for every staged candidate that passes the block cull, hit or not, and the split would triple it.  Not measured.
// Why mma.sync and not tcgen05: as for raster_bwd_wide_mma_kernel, the product is per warp and issued from inside the
// replay loop whose A operand (the weights) the lanes produce a few instructions earlier.
#include "raster_fast.cuh"

namespace gs {

constexpr int kXwBatch = 16;   // staged tile-list entries per buffer
constexpr int kXwWarps = 2;    // warps per CTA (four CTAs per tile, as the wide kernel's default)
constexpr int kXwGroup = 16;   // survivors per tensor-core product (M of the mma)
constexpr int kXwWS = 36;      // row stride of the weight tile (float2 units): conflict-free A loads

struct XwideLayout {
  int FP, GS;                        // feature row (multiple of 64), row stride of the G tile (floats)
  size_t stage_bytes, warp_bytes;
  __host__ __device__ explicit XwideLayout(int F)
      : FP(xwide_row(F)), GS(xwide_row(F) + 4), stage_bytes((size_t)2 * kXwBatch * (32 + xwide_row(F) * 4)),
        warp_bytes((size_t)32 * (xwide_row(F) + 4) * 4 + kXwGroup * kXwWS * 8 + kXwGroup * 4) {}
  __host__ __device__ size_t total() const { return stage_bytes + kXwWarps * warp_bytes; }
};

// WGT: the image weight W is differentiable too (gradient gw, forward W in wimg): one more channel whose feature is
// always 1, so RG starts with W_final Gw and G . f_i gains + Gw (see raster_bwd_fast_kernel).
template <bool HEUR, bool WGT = false>
__global__ void __launch_bounds__(kXwWarps * 32)
raster_bwd_xwide_kernel(const __grid_constant__ GsRasterParams p, const float4* __restrict__ rec,
                        const float* __restrict__ featP, const int32_t* __restrict__ ranges,
                        const int32_t* __restrict__ o2p, const float* __restrict__ image,
                        const float* __restrict__ grad_image, float* __restrict__ grad_pts,
                        float* __restrict__ grad_feat, float* __restrict__ heuristic,
                        const float* __restrict__ wimg, const float* __restrict__ gw) {
  constexpr int NG = 7 + (HEUR ? 2 : 0);             // geometry (+ heuristic) values
  constexpr int kThreads = kXwWarps * 32, kParts = 8 / kXwWarps;
  const int F = p.num_features;
  const XwideLayout L(F);
  const int FP = L.FP, GS = L.GS;
  extern __shared__ __align__(16) unsigned char smem[];
  float4* s_r0 = reinterpret_cast<float4*>(smem);                        // [2][kXwBatch]
  float4* s_r1 = s_r0 + 2 * kXwBatch;                                    // [2][kXwBatch]
  float* s_feat = reinterpret_cast<float*>(smem + 2 * kXwBatch * 32);    // [2][kXwBatch][FP]

  const int tile = blockIdx.x / kParts, t = threadIdx.x, lane = t & 31, lwarp = t >> 5;
  const int warp = (blockIdx.x % kParts) * kXwWarps + lwarp;   // which 8x4 pixel block of the tile
  unsigned char* wbase = smem + L.stage_bytes + (size_t)lwarp * L.warp_bytes;
  float* s_G = reinterpret_cast<float*>(wbase);                                        // [32][GS]
  float2* s_W = reinterpret_cast<float2*>(wbase + (size_t)32 * GS * 4);                // [16][WS] {hi, lo}
  int* s_idx = reinterpret_cast<int*>(wbase + (size_t)32 * GS * 4 + kXwGroup * kXwWS * 8);   // [16]

  const int tw = (p.image_width + kFastTile - 1) / kFastTile;
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

  float* my_G = s_G + lane * GS;
  float W = inb ? 0.f : 1.f, RG = 0.f, Gw = 0.f;
  {
    const int64_t pix = (int64_t)py * p.image_width + px;   // 64 bit: a 4K image of 256 channels has 2.1 G elements
#pragma unroll 4
    for (int c = 0; c < FP; ++c) {
      const bool ok = inb && c < F;
      const float g = ok ? grad_image[pix * F + c] : 0.f;
      RG = fmaf(ok ? image[pix * F + c] : 0.f, g, RG);
      my_G[c] = g;
    }
    if constexpr (WGT) {
      Gw = inb ? gw[pix] : 0.f;
      RG = fmaf(inb ? wimg[pix] : 0.f, Gw, RG);
    }
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
        const float2 a0 = s_W[gid * kXwWS + tig + 8 * k], a1 = s_W[(gid + 8) * kXwWS + tig + 8 * k];
        const float2 a2 = s_W[gid * kXwWS + tig + 4 + 8 * k], a3 = s_W[(gid + 8) * kXwWS + tig + 4 + 8 * k];
        ahi[k][0] = __float_as_uint(a0.x); ahi[k][1] = __float_as_uint(a1.x);
        ahi[k][2] = __float_as_uint(a2.x); ahi[k][3] = __float_as_uint(a3.x);
        alo[k][0] = __float_as_uint(a0.y); alo[k][1] = __float_as_uint(a1.y);
        alo[k][2] = __float_as_uint(a2.y); alo[k][3] = __float_as_uint(a3.y);
      }
      const int s0 = gid, s1 = gid + 8;
      const int64_t i0 = s0 < ns ? s_idx[s0] : -1, i1 = s1 < ns ? s_idx[s1] : -1;
#pragma unroll 2
      for (int n = 0; n < FP / 8; ++n) {
        float c[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float b0 = s_G[(tig + 8 * k) * GS + gid + 8 * n], b1 = s_G[(tig + 4 + 8 * k) * GS + gid + 8 * n];
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
  const int nb = (C + kXwBatch - 1) / kXwBatch;

  auto issue_load = [&](int b) {
    const int buf = b & 1;
    if (t < kXwBatch) {
      const int v = b * kXwBatch + t;
      if (v < C) {
        const int idx = o2p[start + v];
        cp_async16(&s_r0[buf * kXwBatch + t], rec + 2 * (int64_t)idx);
        cp_async16(&s_r1[buf * kXwBatch + t], rec + 2 * (int64_t)idx + 1);
      }
    }
    const int CH = FP / 4;
    for (int q = t; q < kXwBatch * CH; q += kThreads) {
      const int slot = q / CH, part = q - slot * CH;
      const int v = b * kXwBatch + slot;
      if (v < C) {
        const int idx = o2p[start + v];
        cp_async16(s_feat + ((size_t)buf * kXwBatch + slot) * FP + part * 4, featP + (int64_t)idx * FP + part * 4);
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
    const int n_in = min(kXwBatch, C - b * kXwBatch);
    if (!warp_done) {
      bool touch = false;
      if (lane < n_in) {
        const float4 r0 = s_r0[buf * kXwBatch + lane], r1 = s_r1[buf * kXwBatch + lane];
        const float cx = kSqrtHalfLog2e * r1.x, cy = kSqrtHalfLog2e * r1.y;
        touch = block_may_touch(r0.x, r0.y, r0.z * cx, r0.w * cx, -r0.w * cy, r0.z * cy, log2f(r1.z) - l2thr, bx0, bx1,
                                by0, by1);
      }
      unsigned mask = __ballot_sync(kFull, touch);
      while (mask) {
        const int j = __ffs(mask) - 1;
        mask &= mask - 1;
        const float4 r0 = s_r0[buf * kXwBatch + j], r1 = s_r1[buf * kXwBatch + j];
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
          // G . f_i over all F channels (padded channels are zero in both)
          const float* frow = s_feat + ((size_t)buf * kXwBatch + j) * FP;
          float fG0 = 0.f, fG1 = 0.f, fG2 = 0.f, fG3 = 0.f;   // four independent chains: the dot product is latency bound
#pragma unroll 4
          for (int c = 0; c < FP; c += 4) {
            const float4 f4 = *reinterpret_cast<const float4*>(frow + c);
            const float4 g4 = *reinterpret_cast<const float4*>(my_G + c);
            fG0 = fmaf(f4.x, g4.x, fG0); fG1 = fmaf(f4.y, g4.y, fG1);
            fG2 = fmaf(f4.z, g4.z, fG2); fG3 = fmaf(f4.w, g4.w, fG3);
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
          s_W[ns * kXwWS + lane] = make_float2(whi, __uint_as_float(tf32_rna(wl - whi)));
          if (lane == 0) s_idx[ns] = (int)idx;
          if (++ns == kXwGroup) flush_group();
        }
      }
      warp_done = __all_sync(kFull, W >= sat);
    }
    if (__syncthreads_and(warp_done)) break;
  }
  cp_async_wait<0>();
  if (ns > 0) flush_group();
}

template <bool HEUR, bool WGT>
static int launch_xwide(const GsRasterParams& p, const RasterArgs& a, const float4* rec, const float* featP,
                        cudaStream_t st) {
  const size_t smem = XwideLayout(p.num_features).total();
  const int tiles = tiles_wide(p) * tiles_high(p);
  // per launch: the attribute belongs to the (function, device) pair and the call costs about a microsecond
  GS_CUDA(cudaFuncSetAttribute(raster_bwd_xwide_kernel<HEUR, WGT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)smem));
  raster_bwd_xwide_kernel<HEUR, WGT><<<tiles * (8 / kXwWarps), kXwWarps * 32, smem, st>>>(
      p, rec, featP, a.tile_ranges, a.overlap_to_point, (const float*)a.image_in, (const float*)a.grad_image,
      (float*)a.grad_gaussians, (float*)a.grad_features, HEUR ? (float*)a.point_heuristic : nullptr,
      (const float*)a.image_weight, (const float*)a.grad_image_weight);
  GS_LAUNCH_CHECK();
  return GS_OK;
}

int raster_bwd_xwide(const GsRasterParams& p, const RasterArgs& a, const float4* rec, const float* featP,
                     cudaStream_t st) {
  const bool heur = p.compute_point_heuristic && a.point_heuristic != nullptr;
  if (a.grad_image_weight != nullptr)
    return heur ? launch_xwide<true, true>(p, a, rec, featP, st) : launch_xwide<false, true>(p, a, rec, featP, st);
  return heur ? launch_xwide<true, false>(p, a, rec, featP, st) : launch_xwide<false, false>(p, a, rec, featP, st);
}

}  // namespace gs
