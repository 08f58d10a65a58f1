// raster_fast_fwd.cu — forward rasterizer, f32 / alpha blending / tile 16 (the measured path).
//
// Replaces rasterizer/forward.py:24-137 of /root/reference/taichi_splatting/.  Same per pixel arithmetic
// (front-to-back blend in depth order, weight = alpha (1 - W), alpha = min(alpha0 p, clamp) tested against
// alpha_threshold), different machine mapping:
//   * one CTA per 16x16 tile, 8 warps, each warp owns an 8x4 pixel block (one pixel per lane);
//   * the tile's sorted gaussians are staged in batches of 128 through shared memory with cp.async
//     (16 B gathers of pre-packed 32 B records + padded feature rows), double buffered;
//   * raster_cull_mask_kernel tests every tile-list entry ONCE per frame against the eight 8x4 pixel blocks of
//     its tile (exact minimum of the ellipse's quadratic form over the block) and leaves a byte per entry; the
//     byte is staged with the entry, each warp gathers its bit into ballot masks and only walks the survivors —
//     a gaussian that cannot pass alpha_threshold anywhere in the block contributes exactly nothing, so results
//     do not change, but most (warp, gaussian) pairs of a tile list vanish (the test used to run in every warp
//     of both rasterizer passes: 17 % of the forward's instructions);
//   * exp via ex2.approx on a pre-scaled exponent (alpha = 2^(log2 alpha0 - |M d|^2));
//   * a warp stops when every lane's transmittance is <= forward_exit_transmittance (0 = exact: no
//     later term can change anything); the CTA stops when all warps have;
//   * the reference's stale-slot re-read (forward.py:88, SURVEY Q1) is reproduced, when requested, by
//     re-walking entries [C-256, (G-1) 256) after the C real ones with visibility recording off.
#include "raster_fast.cuh"

namespace gs {

constexpr int kFwdThreads = 256;

// ------------------------------------------------------------------------------------------------ pack
template <int FP>
__global__ void __launch_bounds__(256)
raster_pack_kernel(int64_t V, int F, const float* __restrict__ g, const float* __restrict__ feat,
                   float4* __restrict__ recF, float* __restrict__ featP, float4* __restrict__ recB) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= V) return;
  const float* gi = g + 7 * i;
  const float mx = gi[0], my = gi[1], ax = gi[2], ay = gi[3], sx = gi[4], sy = gi[5], alpha = gi[6];
  const float isx = 1.0f / sx, isy = 1.0f / sy;
  if (recF) {
    const float cx = kSqrtHalfLog2e * isx, cy = kSqrtHalfLog2e * isy;
    recF[2 * i] = make_float4(mx, my, ax * cx, ay * cx);
    recF[2 * i + 1] = make_float4(-ay * cy, ax * cy, log2f(alpha), __int_as_float((int)i));
  }
  if (recB) {
    recB[2 * i] = make_float4(mx, my, ax, ay);
    recB[2 * i + 1] = make_float4(isx, isy, alpha, __int_as_float((int)i));
  }
  if (featP) {
    float f[FP];
#pragma unroll
    for (int c = 0; c < FP; ++c) f[c] = c < F ? feat[i * F + c] : 0.f;
#pragma unroll
    for (int c = 0; c < FP; c += 4)
      *reinterpret_cast<float4*>(featP + i * FP + c) = make_float4(f[c], f[c + 1], f[c + 2], f[c + 3]);
  }
}

// extra-wide features whose rows are not a whole number of 64-channel slices, and bf16 rows that are not a whole
// number of 8-channel chunks: one thread per padded element
template <typename TF>
__global__ void __launch_bounds__(256)
raster_pad_rows_kernel(int64_t n, int F, int FP, const TF* __restrict__ feat, TF* __restrict__ featP) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= n) return;
  const int64_t i = q / FP;
  const int c = (int)(q - i * FP);
  featP[q] = c < F ? feat[i * F + c] : TF();
}

int raster_fast_pack(const GsRasterParams& p, const RasterArgs& a, bool forward, bool features, cudaStream_t st) {
  if (p.num_points == 0) return GS_OK;
  // extra-wide or bf16 features (8..256 channels): records as for the wide path, features padded to 64-channel slices
  // (extra-wide) or to bf16_feature_pad
  if (xwide_features(p.num_features) || p.dtype == GS_BF16) {
    const FastLayout L = fast_layout(p);
    if (L.feat_in_place && ((uintptr_t)a.features & 15) != 0) {   // cp.async stages them in 16 B pieces
      set_error("rasterizer: %d feature channels are read in place and must be 16-byte aligned", p.num_features);
      return GS_ERR_INVALID;
    }
    unsigned char* ws = (unsigned char*)a.workspace;
    const bool want_bwd = !forward || p.points_requires_grad || p.features_requires_grad;
    raster_pack_kernel<4><<<(unsigned)ceil_div(p.num_points, 256), 256, 0, st>>>(
        p.num_points, p.num_features, (const float*)a.gaussians2d, nullptr, forward ? (float4*)(ws + L.off_recF) : nullptr,
        nullptr, want_bwd ? (float4*)(ws + L.off_recB) : nullptr);
    GS_LAUNCH_CHECK();
    if (features && !L.feat_in_place) {
      const int64_t n = p.num_points * (int64_t)L.FP;
      if (p.dtype == GS_BF16)
        raster_pad_rows_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(
            n, p.num_features, L.FP, (const __nv_bfloat16*)a.features, (__nv_bfloat16*)(ws + L.off_feat));
      else
        raster_pad_rows_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(n, p.num_features, L.FP, (const float*)a.features,
                                                                           (float*)(ws + L.off_feat));
      GS_LAUNCH_CHECK();
    }
    return GS_OK;
  }
  const FastLayout L = fast_layout(p);
  unsigned char* ws = (unsigned char*)a.workspace;
  // the forward call also packs the backward records when a gradient will be asked for, so that the backward
  // call (workspace_holds_packed) launches no pack kernel at all
  // The narrow backward (F <= 7, raster_fast_bwd.cu) walks the forward's records; only the wide one has its own.
  // Antialiased rendering (narrow features only) walks the unscaled records {mean, axis}{1/sigma, alpha, index} in
  // both passes: its per pixel function needs the axis and the sigmas separately.
  const bool want_bwd = !forward || p.points_requires_grad || p.features_requires_grad;
  const bool narrow = p.num_features <= 7;
  float4* recF = (!p.antialias && (forward || narrow)) ? (float4*)(ws + L.off_recF) : nullptr;
  float4* recB = (p.antialias || (want_bwd && !narrow)) ? (float4*)(ws + L.off_recB) : nullptr;
  float* featP = features ? (float*)(ws + L.off_feat) : nullptr;
  const int64_t blocks = ceil_div(p.num_points, 256);
#define GS_PACK(FPV)                                                                                          \
  raster_pack_kernel<FPV><<<(unsigned)blocks, 256, 0, st>>>(p.num_points, p.num_features, (const float*)a.gaussians2d, \
                                                            (const float*)a.features, recF, featP, recB)
  switch (L.FP) {
    case 4: GS_PACK(4); break;
    case 8: GS_PACK(8); break;
    case 16: GS_PACK(16); break;
    case 36: GS_PACK(36); break;
    default: GS_PACK(64); break;
  }
#undef GS_PACK
  GS_LAUNCH_CHECK();
  return GS_OK;
}

// ------------------------------------------------------------------------------------------------ cull masks
// One pass over the tile lists: entry k of tile t gets a byte whose bit w says whether the gaussian can pass
// alpha_threshold anywhere in the 8x4 pixel block w of the tile (w = 2 * block row + block column; exact minimum of
// the ellipse's quadratic form over the block, with the slack of block_may_touch).  The forward (eight warps, one block
// each) and the narrow backward (two warps, four blocks each) read the byte instead of repeating the test per warp.
// AA: antialiased rendering evaluates the gaussian INTEGRATED over the pixel (raster_math.cuh pdf_aa: the pixel's unit
// box in the gaussian's frame), which is bounded by the maximum of the point-sampled gaussian over that box: the same
// test on the block grown by the box's half diagonal (0.75 px covers it) and with a factor two of slack on alpha for
// the logistic approximation of the normal CDF is conservative.  Records there are {mean, axis}{1/sigma, alpha, index}.
template <bool AA>
__global__ void __launch_bounds__(128)
raster_cull_mask_kernel(const __grid_constant__ GsRasterParams p, const float4* __restrict__ rec,
                        const int32_t* __restrict__ ranges, const int32_t* __restrict__ o2p,
                        unsigned char* __restrict__ mask) {
  const int tile = blockIdx.x;
  const int tw = (p.image_width + kFastTile - 1) / kFastTile;
  const float grow = AA ? 0.75f : 0.f;
  const float x0 = (float)((tile % tw) * kFastTile) + 0.5f - grow, y0 = (float)((tile / tw) * kFastTile) + 0.5f - grow;
  const float l2thr = log2f((float)p.alpha_threshold);
  const int start = ranges[2 * tile], end = ranges[2 * tile + 1];
  for (int k = start + threadIdx.x; k < end; k += blockDim.x) {
    const int idx = o2p[k];
    const float4 r0 = rec[2 * (int64_t)idx], r1 = rec[2 * (int64_t)idx + 1];
    float a1x, a1y, a2x, a2y, l2a;
    if (AA) {
      const float cx = kSqrtHalfLog2e * r1.x, cy = kSqrtHalfLog2e * r1.y;
      a1x = r0.z * cx; a1y = r0.w * cx; a2x = -r0.w * cy; a2y = r0.z * cy;
      l2a = log2f(r1.z) + 1.0f;
    } else {
      a1x = r0.z; a1y = r0.w; a2x = r1.x; a2y = r1.y; l2a = r1.z;
    }
    const float A00 = a1x * a1x + a2x * a2x, A01 = a1x * a1y + a2x * a2y, A11 = a1y * a1y + a2y * a2y;
    const float n01r11 = -A01 * fast_rcp(A11), n01r00 = -A01 * fast_rcp(A00);
    const float qlim = (l2a - l2thr) * 1.001f + 1e-3f;
    unsigned bits = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      const float dx0 = x0 + (float)((w & 1) * 8) - r0.x, dx1 = dx0 + 7.f + 2.f * grow;
      const float dy0 = y0 + (float)((w >> 1) * 4) - r0.y, dy1 = dy0 + 3.f + 2.f * grow;
      const float dxc = fminf(fmaxf(0.f, dx0), dx1), dyc = fminf(fmaxf(0.f, dy0), dy1);
      const float dyv = fminf(fmaxf(n01r11 * dxc, dy0), dy1);
      const float qv = A00 * dxc * dxc + 2.f * A01 * dxc * dyv + A11 * dyv * dyv;
      const float dxh = fminf(fmaxf(n01r00 * dyc, dx0), dx1);
      const float qh = A00 * dxh * dxh + 2.f * A01 * dxh * dyc + A11 * dyc * dyc;
      bits |= (fminf(qv, qh) < qlim ? 1u : 0u) << w;
    }
    mask[k] = (unsigned char)bits;
  }
}

int raster_cull_mask(const GsRasterParams& p, const RasterArgs& a, cudaStream_t st) {
  if (p.num_overlaps == 0) return GS_OK;
  const FastLayout L = fast_layout(p);
  unsigned char* ws = (unsigned char*)a.workspace;
  const int tiles = tiles_wide(p) * tiles_high(p);
  if (p.antialias)
    raster_cull_mask_kernel<true><<<tiles, 128, 0, st>>>(p, (const float4*)(ws + L.off_recB), a.tile_ranges,
                                                         a.overlap_to_point, ws + L.off_mask);
  else
    raster_cull_mask_kernel<false><<<tiles, 128, 0, st>>>(p, (const float4*)(ws + L.off_recF), a.tile_ranges,
                                                          a.overlap_to_point, ws + L.off_mask);
  GS_LAUNCH_CHECK();
  return GS_OK;
}

// ------------------------------------------------------------------------------------------------ forward
// BATCH = staged tile-list entries per buffer: 128 for narrow features, 64 for FP >= 16 (shared memory budget).
// FOURTH: with FP = 4 the fourth accumulator is only needed when F = 4 (it is padding for F <= 3).
// XW: extra-wide features (65..256 channels).  The CTA of blockIdx.y = s blends channel slice [64 s, 64 s + 64) of
// rows of xwide_row(F) floats; every slice walks the tile list with the same records, cull bytes and exit test, and
// only slice 0 writes image_alpha and visibility.  Why CTAs per slice and not slice warps inside one CTA: a tile's
// 256 pixels x 256 channels of accumulators (256 KB) are the whole register file of an SM, so a CTA can hold the
// full channel range of a few pixel blocks only, and each such CTA would stage all F channels of every entry (4 x
// the feature bytes at F = 256 for four CTAs per tile); a slice CTA stages its own 64 channels and the records.
// TF: feature / image storage (float, or __nv_bfloat16 for GS_BF16: rows of FP = 8, 16, 40, 64 bf16, or 64-channel
// slices; each feature is widened to f32 where it is used, the blend is the f32 one, the image is rounded once).
template <int FP, bool VIS, int BATCH, bool FOURTH = true, bool AA = false, bool XW = false, typename TF = float>
__global__ void __launch_bounds__(kFwdThreads, FP <= 8 ? 0 : (FP <= 40 ? 4 : 2))   // narrow: no occupancy target (the compiler settles on 30 registers = 8 CTAs per SM by itself; forcing 8 lengthened the VIS walk); 64 / 128 registers for the wide ones
raster_fwd_fast_kernel(const __grid_constant__ GsRasterParams p, const float4* __restrict__ rec,
                       const TF* __restrict__ featP, const int32_t* __restrict__ ranges,
                       const int32_t* __restrict__ o2p, TF* __restrict__ image, float* __restrict__ image_alpha,
                       float* __restrict__ visibility, const unsigned char* __restrict__ cull_mask) {
  constexpr int kFwdBatch = BATCH;
  constexpr int CE = kChunkElems<TF>;   // features per 16 B unit: 4 f32 or 8 bf16
  // one staged entry = {record (2 x float4), feature row (FP / CE 16 B units)} in consecutive 16 B units: one address
  // per entry in the inner loop.  U is odd so that a lane-per-entry LDS.128 (the cull) is bank-conflict free (bf16:
  // U = 3, 5, 7, 11 for FP = 8, 16, 40, 64).
  constexpr int U = (2 + FP / CE) | 1;
  __shared__ __align__(16) float4 s_e[2][kFwdBatch][U];
  __shared__ unsigned char s_mask[2][kFwdBatch];   // cull bytes of the staged entries (raster_cull_mask_kernel)
  // VIS: the visibility sums of every staged entry, one word per warp (23 bit fixed point: 32 pixels stay below 2^28),
  // merged over the eight warps after the batch and committed with ONE global atomic per entry and tile, as the
  // reference's kernel does (rasterizer/forward.py:116-128) — round 1 issued one global atomic per surviving (warp,
  // entry) pair.  Plain stores, no shared-memory atomics: the merging thread clears the words it has read.
  __shared__ __align__(16) unsigned s_vis[VIS ? 2 : 1][VIS ? kFwdBatch : 1][8];

  const int tile = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int tw = (p.image_width + kFastTile - 1) / kFastTile;
  const int F = p.num_features;
  const int wx0 = (tile % tw) * kFastTile + (warp & 1) * 8;
  const int wy0 = (tile / tw) * kFastTile + (warp >> 1) * 4;
  const int px = wx0 + (lane & 7), py = wy0 + (lane >> 3);
  const bool inb = px < p.image_width && py < p.image_height;
  const float pxf = (float)px + 0.5f, pyf = (float)py + 0.5f;
  const float thr = (float)p.alpha_threshold, cmax = (float)p.clamp_max_alpha;
  const float exit_T = (float)p.forward_exit_transmittance;
  // feature row stride and this CTA's first channel (XW), whether it writes image_alpha / visibility
  const int frow = XW ? xwide_row(F) : FP;
  const int c_base = XW ? (int)blockIdx.y * FP : 0;
  const bool first_slice = !XW || blockIdx.y == 0;

  float acc[FP];
#pragma unroll
  for (int c = 0; c < FP; ++c) acc[c] = 0.f;
  float W = inb ? 0.f : 1.f;

  const int start = ranges[2 * tile], end = ranges[2 * tile + 1];
  const int C = end - start;
  const int G = (C + kFastTileArea - 1) / kFastTileArea;
  const int extra = (p.emulate_stale_tail && G > 1) ? (G * kFastTileArea - C) : 0;  // stale slots re-read (Q1)
  const int total = C + extra;
  const int nb = (total + kFwdBatch - 1) / kFwdBatch;

  auto issue_load = [&](int b) {
    const int buf = b & 1;
    if constexpr (BATCH * 2 == kFwdThreads) {  // narrow rows: first half of the CTA gathers records, second half features
      const int slot = t & (kFwdBatch - 1);
      const int v = b * kFwdBatch + slot;
      if (v < total) {
        const int k = v < C ? v : v - kFastTileArea;
        const int idx = o2p[start + k];
        if (t < kFwdBatch) {
          const unsigned char m = cull_mask[start + k];   // in flight together with the index load
          cp_async16(&s_e[buf][slot][0], rec + 2 * (int64_t)idx);
          cp_async16(&s_e[buf][slot][1], rec + 2 * (int64_t)idx + 1);
          s_mask[buf][slot] = m;
        } else {
#pragma unroll
          for (int c = 0; c < FP; c += CE) cp_async16(&s_e[buf][slot][2 + c / CE], featP + (int64_t)idx * frow + c_base + c);
        }
      }
    } else {  // wide rows: records by the first BATCH threads, the 16 B feature chunks spread over the whole CTA
      if (t < kFwdBatch) {
        const int v = b * kFwdBatch + t;
        if (v < total) {
          const int k = v < C ? v : v - kFastTileArea;
          const int idx = o2p[start + k];
          const unsigned char m = cull_mask[start + k];
          cp_async16(&s_e[buf][t][0], rec + 2 * (int64_t)idx);
          cp_async16(&s_e[buf][t][1], rec + 2 * (int64_t)idx + 1);
          s_mask[buf][t] = m;
        }
      }
      constexpr int CH = FP / CE;
#pragma unroll
      for (int q0 = 0; q0 < kFwdBatch * CH; q0 += kFwdThreads) {
        const int q = q0 + t;
        const int slot = q / CH, part = q - slot * CH;
        const int v = b * kFwdBatch + slot;
        if (q < kFwdBatch * CH && v < total) {
          const int idx = o2p[start + (v < C ? v : v - kFastTileArea)];
          cp_async16(&s_e[buf][slot][2 + part], featP + (int64_t)idx * frow + c_base + part * CE);
        }
      }
    }
    cp_async_commit();
  };

  if constexpr (VIS) {   // ordered before the first shared atomic by the barrier of the first batch
    for (int q = t; q < 2 * kFwdBatch * 8; q += kFwdThreads) (&s_vis[0][0][0])[q] = 0u;
  }
  bool warp_done = __all_sync(kFull, (1.f - W) <= exit_T);
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
    const int vbase = b * kFwdBatch;
    const int n_in = min(kFwdBatch, total - vbase);
    if (!warp_done) {
      for (int c0 = 0; c0 < n_in; c0 += 32) {
        const int e = c0 + lane;
        const bool hit = e < n_in && ((s_mask[buf][e] >> warp) & 1u);
        unsigned mask = __ballot_sync(kFull, hit);
        while (mask) {
          const int j = c0 + __ffs(mask) - 1;
          mask &= mask - 1;
          const float4* ent = s_e[buf][j];
          const float4 r0 = ent[0], r1 = ent[1];
          const float dx = pxf - r0.x, dy = pyf - r0.y;
          float alpha;
          if constexpr (AA) {   // gaussian integrated over the pixel: raster_math.cuh pdf_aa with MUFU ex2 / rcp
            const float tx = fmaf(dy, r0.w, dx * r0.z), ty = fmaf(dy, r0.z, -dx * r0.w);
            const float Sx = aa_sig(( tx + 0.5f) * r1.x) - aa_sig((tx - 0.5f) * r1.x);
            const float Sy = aa_sig(( ty + 0.5f) * r1.y) - aa_sig((ty - 0.5f) * r1.y);
            alpha = fminf(6.283185307179586f * r1.z * fast_rcp(r1.x * r1.y) * (Sx * Sy), cmax);
          } else {
            const float tx = fmaf(dy, r0.w, dx * r0.z);
            const float ty = fmaf(dy, r1.y, dx * r1.x);
            const float ex = fmaf(-ty, ty, fmaf(-tx, tx, r1.z));
            alpha = fminf(fast_ex2(ex), cmax);
          }
          // branch-free blend: a pixel below the threshold adds weight 0 (exactly nothing), which costs less than
          // the divergent branch did (the cull leaves few gaussians that miss every pixel of the block)
          const float weight = alpha > thr ? alpha * (1.f - W) : 0.f;
          W += weight;
          if constexpr (kBf16Storage<TF>) {
#pragma unroll
            for (int c8 = 0; c8 < FP / 8; ++c8) {
              const uint4 u = reinterpret_cast<const uint4*>(ent)[2 + c8];
              const unsigned wd[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                acc[8 * c8 + 2 * k] = fmaf(bf16_lo(wd[k]), weight, acc[8 * c8 + 2 * k]);
                acc[8 * c8 + 2 * k + 1] = fmaf(bf16_hi(wd[k]), weight, acc[8 * c8 + 2 * k + 1]);
              }
            }
          } else {
#pragma unroll
            for (int c4 = 0; c4 < FP / 4; ++c4) {
              const float4 f4 = ent[2 + c4];
              acc[4 * c4] = fmaf(f4.x, weight, acc[4 * c4]);
              acc[4 * c4 + 1] = fmaf(f4.y, weight, acc[4 * c4 + 1]);
              acc[4 * c4 + 2] = fmaf(f4.z, weight, acc[4 * c4 + 2]);
              if (FP > 4 || FOURTH) acc[4 * c4 + 3] = fmaf(f4.w, weight, acc[4 * c4 + 3]);
            }
          }
          if constexpr (VIS) {
            // visibility[g] += sum over the tile's pixels of the blend weight.  The weights are in [0, 0.99]: summed as
            // 23 bit fixed point with ONE redux.sync (integer warp reduction) instead of five float shuffles, then one
            // shared-memory atomic per warp.  The fixed-point value is the mantissa of 1 + weight (one FADD rounds the
            // weight to a multiple of 2^-23; no multiply, no float -> integer conversion on the MUFU pipe): the 32
            // exponent fields add up to 32 * 0x3f800000 = 0xf0000000 mod 2^32, taken off after the reduction.  The
            // quantisation (2^-24 per pixel) is far below the f32 rounding of the running sums.  Stale re-reads (Q1,
            // vbase + j >= C: warp-uniform) do not count, as in the reference, whose write-back skips those slots.
            // One predicated store of the warp's sum into the warp's own word: an atomic on a warp-uniform shared address
            // makes ptxas emit its warp-aggregation sequence (vote, leader election, popc, multiply: 9 more instructions
            // per survivor) although a single lane enters.
            const unsigned total_q = __reduce_add_sync(kFull, __float_as_uint(1.0f + weight)) - 0xf0000000u;
            if (lane == 0 && vbase + j < C && first_slice) s_vis[buf][j][warp] = total_q;
          }
        }
      }
      warp_done = __all_sync(kFull, (1.f - W) <= exit_T);
    }
    const bool all_done = __syncthreads_and(warp_done);
    if constexpr (VIS) {
      // the thread that staged slot t (and will stage it again two batches on) commits and clears the slot's sum
      if (t < kFwdBatch) {
        uint4* w4 = reinterpret_cast<uint4*>(&s_vis[buf][t][0]);
        const uint4 a = w4[0], b = w4[1];
        const unsigned q = (a.x + a.y) + (a.z + a.w) + (b.x + b.y) + (b.z + b.w);
        if (q != 0u) {
          w4[0] = make_uint4(0u, 0u, 0u, 0u);
          w4[1] = make_uint4(0u, 0u, 0u, 0u);
          atomicAdd(visibility + __float_as_int(s_e[buf][t][1].w), (float)q * (1.f / 8388608.f));
        }
      }
    }
    if (all_done) break;
  }
  cp_async_wait<0>();

  if (inb) {
    const int64_t pix = (int64_t)py * p.image_width + px;
#pragma unroll
    for (int c = 0; c < FP; ++c)
      if (c_base + c < F) image[pix * F + c_base + c] = from_f32<TF>(acc[c]);
    if (first_slice) image_alpha[pix] = W;
  }
}

bool raster_fast_supported(const GsRasterParams& p) {
  return (p.dtype == GS_F32 || p.dtype == GS_BF16) && p.tile_size == kFastTile && (!p.antialias || p.num_features <= 7) &&
         p.use_alpha_blending && (fast_feature_pad(p.num_features) != 0 || xwide_features(p.num_features)) &&
         p.num_points < (1ll << 31);
}

size_t raster_fast_workspace_bytes(const GsRasterParams& p) { return fast_layout(p).total; }

// GS_BF16 (8..256 channels, no antialiasing): the f32 kernel's modes instantiated over bf16 rows
static int raster_fwd_fast_bf16(const GsRasterParams& p, const RasterArgs& a, const float4* rec,
                                const __nv_bfloat16* featP, const unsigned char* cmask, bool vis, cudaStream_t st) {
  using bf16 = __nv_bfloat16;
  const FastLayout L = fast_layout(p);
  const int tiles = tiles_wide(p) * tiles_high(p);
  if (xwide_features(p.num_features)) {   // one CTA per (tile, 64-channel slice)
    const dim3 grid(tiles, L.FP / kXwideSlice);
#define GS_FWD_XW16(VISV)                                                                                          \
  raster_fwd_fast_kernel<kXwideSlice, VISV, 64, true, false, true, bf16><<<grid, kFwdThreads, 0, st>>>(            \
      p, rec, featP, a.tile_ranges, a.overlap_to_point, (bf16*)a.image, (float*)a.image_alpha, (float*)a.visibility, \
      cmask)
    if (vis) GS_FWD_XW16(true); else GS_FWD_XW16(false);
#undef GS_FWD_XW16
    GS_LAUNCH_CHECK();
    return GS_OK;
  }
#define GS_FWD_LAUNCH16(FPV, VISV, BATCHV)                                                                         \
  GS_CUDA(launch_background(raster_fwd_fast_kernel<FPV, VISV, BATCHV, true, false, false, bf16>, dim3(tiles),     \
                            dim3(kFwdThreads), 0, st, p, rec, featP, a.tile_ranges, a.overlap_to_point,           \
                            (bf16*)a.image, (float*)a.image_alpha, (float*)a.visibility, cmask))
#define GS_FWD_CASE16(FPV, BATCHV) \
  case FPV: if (vis) GS_FWD_LAUNCH16(FPV, true, BATCHV); else GS_FWD_LAUNCH16(FPV, false, BATCHV); break
  switch (L.FP) {
    GS_FWD_CASE16(8, 128);
    GS_FWD_CASE16(16, 64);
    GS_FWD_CASE16(40, 64);
    GS_FWD_CASE16(64, 64);
    default: GS_UNSUPPORTED("rasterizer forward (bf16): %d feature channels", p.num_features);
  }
#undef GS_FWD_CASE16
#undef GS_FWD_LAUNCH16
  GS_LAUNCH_CHECK();
  return GS_OK;
}

int raster_fwd_fast(const GsRasterParams& p, const RasterArgs& a, cudaStream_t st) {
  int rc = raster_fast_pack(p, a, /*forward=*/true, /*features=*/true, st);
  if (rc != GS_OK) return rc;
  rc = raster_cull_mask(p, a, st);
  if (rc != GS_OK) return rc;
  const FastLayout L = fast_layout(p);
  unsigned char* ws = (unsigned char*)a.workspace;
  const unsigned char* cmask = ws + L.off_mask;
  const float4* rec = (const float4*)(ws + (p.antialias ? L.off_recB : L.off_recF));
  const int tiles = tiles_wide(p) * tiles_high(p);
  const bool vis = p.compute_visibility && a.visibility != nullptr;
  if (p.dtype == GS_BF16)
    return raster_fwd_fast_bf16(p, a, rec, (const __nv_bfloat16*)fast_feature_rows(p, a), cmask, vis, st);
  const float* featP = (const float*)fast_feature_rows(p, a);
  if (xwide_features(p.num_features)) {   // one CTA per (tile, 64-channel slice)
    const dim3 grid(tiles, L.FP / kXwideSlice);
#define GS_FWD_XW(VISV)                                                                                            \
  raster_fwd_fast_kernel<kXwideSlice, VISV, 64, true, false, true><<<grid, kFwdThreads, 0, st>>>(                  \
      p, rec, featP, a.tile_ranges, a.overlap_to_point, (float*)a.image, (float*)a.image_alpha, (float*)a.visibility, \
      cmask)
    if (vis) GS_FWD_XW(true); else GS_FWD_XW(false);
#undef GS_FWD_XW
    GS_LAUNCH_CHECK();
    return GS_OK;
  }
  if (p.antialias) {   // narrow features only (raster_fast_supported)
#define GS_FWD_AA(FPV, VISV, FOURTHV)                                                                              \
  raster_fwd_fast_kernel<FPV, VISV, 128, FOURTHV, true><<<tiles, kFwdThreads, 0, st>>>(                            \
      p, rec, featP, a.tile_ranges, a.overlap_to_point, (float*)a.image, (float*)a.image_alpha,                    \
      (float*)a.visibility, cmask)
    if (L.FP == 4 && p.num_features < 4) { if (vis) GS_FWD_AA(4, true, false); else GS_FWD_AA(4, false, false); }
    else if (L.FP == 4) { if (vis) GS_FWD_AA(4, true, true); else GS_FWD_AA(4, false, true); }
    else { if (vis) GS_FWD_AA(8, true, true); else GS_FWD_AA(8, false, true); }
#undef GS_FWD_AA
    GS_LAUNCH_CHECK();
    return GS_OK;
  }
#define GS_FWD_LAUNCH1(FPV, VISV, BATCHV, FOURTHV)                                                                 \
  GS_CUDA(launch_background(raster_fwd_fast_kernel<FPV, VISV, BATCHV, FOURTHV, false>, dim3(tiles), dim3(kFwdThreads), \
                            0, st, p, rec, featP, a.tile_ranges, a.overlap_to_point, (float*)a.image,                \
                            (float*)a.image_alpha, (float*)a.visibility, cmask))
#define GS_FWD_LAUNCH(FPV, VISV, BATCHV)                                                                           \
  do {                                                                                                             \
    if (FPV == 4 && p.num_features < 4) GS_FWD_LAUNCH1(FPV, VISV, BATCHV, false);                                  \
    else GS_FWD_LAUNCH1(FPV, VISV, BATCHV, true);                                                                  \
  } while (0)
#define GS_FWD_CASE(FPV, BATCHV) \
  case FPV: if (vis) GS_FWD_LAUNCH(FPV, true, BATCHV); else GS_FWD_LAUNCH(FPV, false, BATCHV); break
  switch (L.FP) {
    GS_FWD_CASE(4, 128);
    GS_FWD_CASE(8, 128);
    GS_FWD_CASE(16, 64);
    GS_FWD_CASE(36, 64);
    GS_FWD_CASE(64, 64);
    default: GS_UNSUPPORTED("rasterizer forward (fast): %d feature channels", p.num_features);
  }
#undef GS_FWD_CASE
#undef GS_FWD_LAUNCH
#undef GS_FWD_LAUNCH1
  GS_LAUNCH_CHECK();
  return GS_OK;
}

}  // namespace gs
