// raster_fast_bwd.cu — backward rasterizer, f32 / alpha blending / tile 16 (the measured path).
//
// Replaces rasterizer/backward.py:52-228 of /root/reference/taichi_splatting/.  Same per pixel arithmetic:
// front-to-back replay that subtracts each blended term from the final forward image (R -= f w),
// dL/dalpha = sum_c (f_c T - R_c / (1 - alpha)) G_c, threshold tested on the unclamped alpha and gradient
// passed through the clamp (SURVEY Q3), pixels stop at saturate_threshold.  Machine mapping:
//   * one CTA per 16x16 tile, 2 warps; a warp owns a 16x8 region made of four 8x4 sub-blocks and a lane owns the
//     same pixel of each sub-block, so a splat that reaches one or two sub-blocks costs one or two evaluations
//     per lane instead of four (the reference's 2x2 quads always pay four);
//   * cp.async double-buffered staging of 32 B records + padded feature rows, batches of 64;
//   * cull: raster_cull_mask_kernel (raster_fast_fwd.cu) has tested every tile-list entry against the eight 8x4
//     blocks of its tile once per frame (exact minimum of the ellipse's quadratic form over the block); the byte
//     is staged with the entry and turned into four ballot masks; a sub-block is evaluated only if its bit is set
//     (warp-uniform branch);
//   * per pixel state is {W, G_c, RG = sum_c R_c G_c}: the replay needs the remaining features only through R . G
//     (dL/dalpha = T (f . G) - (R . G) / (1 - alpha), and R_c -= f_c w  <=>  RG -= (f . G) w), which halves the
//     per hit arithmetic and the register state compared with carrying R_c;
//   * the geometry gradient of a gaussian is linear in six moments of g = dL/dalpha . p over its pixels, taken in
//     the gaussian's own frame (u, w = offset along / across the axis): sum g, g u, g w, g u^2, g w^2, g u w.  The
//     pixel loop accumulates those (9 instructions per hit instead of 17 for the seven gradient components) and
//     raster_bwd_moments_kernel turns them into d/d(mean, axis, sigma, alpha) once per gaussian afterwards, in
//     place in grad_gaussians;
//   * the 6 + F (+2) per gaussian partial sums are reduced across the warp with a transposed butterfly (12 shuffles
//     for 9 values instead of 45); the lanes that end up owning a value issue one red.global.add each — one
//     reduction per (gaussian, warp), no shared-memory atomics and no block barrier inside the batch.
// A gaussian-parallel "hit record" variant (records appended to shared memory, one lane per gaussian folding
// them, no shuffles) was built and measured in round 1: same instruction count, lower issue rate (1.74 vs 1.58 ms
// on the bench workload), so it was dropped (DESIGN.md, kernel table).
// F is a template parameter (1..7 here, wider F takes raster_generic.cu).
#include "raster_fast.cuh"

namespace gs {


// One warp per CTA, two CTAs per tile: a warp owns a 16x8 region = NSUB = 4 sub-blocks of 8x4 pixels, lane l owns pixel
// (l & 7, l >> 3) of every sub-block, stages the tile list for itself and never waits for its neighbour at a block
// barrier (measured against two warps per CTA and one warp per tile in round 1, see DESIGN.md).
// PAIR: survivors are reduced two at a time — one transposed butterfly over 2 NV values (every exchange step halves
// the live values, so 18 values cost 9 + 5 + 3 + 2 + 1 shuffles where two separate reductions of 9 cost 2 x 12) and
// one red.global.add instruction with 2 NV owning lanes; an odd survivor left at the end of the tile is reduced alone.
// AA: antialiased pixel function (raster_math.cuh pdf_aa_grad with MUFU arithmetic): the records are the unscaled
// {mean, axis}{1/sigma, alpha, index}, the seven gradient components are accumulated directly (the moment trick needs
// a pure gaussian) and no moment pass follows.
// WGT: the image weight W = sum_i w_i is differentiable too (gradient gw (H, W), forward W in wimg).  W is the blend of
// a constant feature 1, so it enters the replay as one more channel: RG starts with W_final Gw and f . G gains + Gw.
template <int F, int FP, bool HEUR, bool PAIR, bool AA = false, bool WGT = false>
__global__ void __launch_bounds__(32, PAIR ? 32 : 1)
raster_bwd_fast_kernel(const __grid_constant__ GsRasterParams p, const float4* __restrict__ rec,
                       const float* __restrict__ featP, const int32_t* __restrict__ ranges,
                       const int32_t* __restrict__ o2p, const float* __restrict__ image,
                       const float* __restrict__ grad_image, float* __restrict__ grad_pts,
                       float* __restrict__ grad_feat, float* __restrict__ heuristic,
                       const unsigned char* __restrict__ cull_mask, const float3 kf,
                       const float* __restrict__ wimg, const float* __restrict__ gw) {
  constexpr int NSUB = 4;
  constexpr int kBwdBatch = 64;   // staged tile-list entries per buffer (32 / 128 measured slower)
  constexpr int NM = AA ? 7 : 6;  // moments: g, g u, g w, g u^2, g w^2, g u w; AA: d/d(mean, axis, sigma, alpha)
  constexpr int NV = NM + F + (HEUR ? 2 : 0);
  // one staged entry = {record (2 x float4), feature row (FP / 4 x float4)} in consecutive 16 B units: one address per
  // entry in the walk (all reads are warp-uniform, so the stride needs no padding)
  constexpr int U = 2 + FP / 4;
  __shared__ __align__(16) float4 s_e[2][kBwdBatch][U];
  __shared__ unsigned char s_mask[2][kBwdBatch];   // cull bytes of the staged entries (raster_cull_mask_kernel)

  const int lane = threadIdx.x;
  const int tile = blockIdx.x >> 1, warp = blockIdx.x & 1;
  const int tw = (p.image_width + kFastTile - 1) / kFastTile;
  const int ox = (tile % tw) * kFastTile, oy = (tile / tw) * kFastTile + warp * (NSUB * 2);
  const int x0 = ox + (lane & 7), y0 = oy + (lane >> 3);
  const float px0 = (float)x0 + 0.5f, py0 = (float)y0 + 0.5f;
  // {alpha_threshold, clamp_max_alpha, saturate_threshold} converted to f32 on the host: as kernel parameters they are
  // constant-bank operands of the compares.  Converted here from the doubles of GsRasterParams, the 64-register cap of
  // the paired variant made the compiler re-issue the F2F.F32.F64 conversions inside the walk (26 of them in the SASS,
  // 3.4 % of the executed instructions, on the MUFU pipe).
  const float thr = kf.x, cmax = kf.y, sat = kf.z;

  // which reduced value this lane commits, and where: value `own` of a single reduction; in a paired reduction values
  // 0 .. NV-1 belong to the first gaussian of the pair and NV .. 2 NV-1 to the second
  auto owner_target = [&](int own, float*& base, unsigned& stride) {
    base = nullptr; stride = 0;   // element offsets stay below 2^31 (raster_fast_supported caps the point count)
    if (own >= 0 && own < NM) {
      if (p.points_requires_grad && grad_pts != nullptr) { base = grad_pts + own; stride = 7; }
    } else if (own >= NM && own < NM + F) {
      if (p.features_requires_grad && grad_feat != nullptr) { base = grad_feat + (own - NM); stride = F; }
    } else if (HEUR && own >= NM + F && own < NV) {
      base = heuristic + (own - NM - F); stride = 2;
    }
  };
  float* own_base; unsigned own_stride;
  owner_target(reduce_owner<NV>(lane), own_base, own_stride);
  float* pair_base = nullptr; unsigned pair_stride = 0; bool pair_second = false;
  if constexpr (PAIR) {
    const int own2 = reduce_owner<2 * NV>(lane);
    pair_second = own2 >= NV;
    owner_target(own2 < 0 ? -1 : (pair_second ? own2 - NV : own2), pair_base, pair_stride);
  }

  // Per pixel state: W, the image gradient G and RG = sum_c R_c G_c.  The replay only ever needs the remaining
  // features R through R . G (dL/dalpha = T (f . G) - (R . G) / (1 - alpha)), and R_c -= f_c w means RG -= (f . G) w.
  float W[NSUB], RG[NSUB], Gd[NSUB][F];
  float Gw[WGT ? NSUB : 1];
#pragma unroll
  for (int i = 0; i < NSUB; ++i) {
    const int px = x0 + 8 * (i & 1), py = y0 + 4 * (i >> 1);
    const bool inb = px < p.image_width && py < p.image_height;
    W[i] = inb ? 0.f : 1.f;
    RG[i] = 0.f;
    const int64_t pix = (int64_t)py * p.image_width + px;
#pragma unroll
    for (int c = 0; c < F; ++c) {
      Gd[i][c] = inb ? grad_image[pix * F + c] : 0.f;
      RG[i] = fmaf(inb ? image[pix * F + c] : 0.f, Gd[i][c], RG[i]);
    }
    if constexpr (WGT) {
      Gw[i] = inb ? gw[pix] : 0.f;
      RG[i] = fmaf(inb ? wimg[pix] : 0.f, Gw[i], RG[i]);
    }
  }

  const int start = ranges[2 * tile], end = ranges[2 * tile + 1];
  const int C = end - start;
  const int nb = (C + kBwdBatch - 1) / kBwdBatch;

  auto issue_load = [&](int b) {
    const int buf = b & 1;
#pragma unroll
    for (int s = lane; s < kBwdBatch; s += 32) {
      const int v = b * kBwdBatch + s;
      if (v < C) {
        const int idx = o2p[start + v];
        const unsigned char m = cull_mask[start + v];   // in flight together with the index load
        cp_async16(&s_e[buf][s][0], rec + 2 * (int64_t)idx);
        cp_async16(&s_e[buf][s][1], rec + 2 * (int64_t)idx + 1);
#pragma unroll
        for (int c = 0; c < FP; c += 4) cp_async16(&s_e[buf][s][2 + c / 4], featP + (int64_t)idx * FP + c);
        s_mask[buf][s] = m;
      }
    }
    cp_async_commit();
  };

  // One survivor: the partial sums of this lane's (up to four) pixels in v[0 .. NV), the gaussian's index returned.
  // bm[i] bit jl = sub-block i can be reached at all (warp-uniform).
  auto evaluate = [&](const float4* ent, const unsigned (&bm)[NSUB], int jl, float* v) -> unsigned {
    const float4 r0 = ent[0], r1 = ent[1];
    float f[F];
#pragma unroll
    for (int c = 0; c < F; ++c) f[c] = reinterpret_cast<const float*>(ent + 2)[c];
    float gf[F];
#pragma unroll
    for (int c = 0; c < F; ++c) gf[c] = 0.f;
    float h0 = 0.f, h1 = 0.f;
    const float dxb = px0 - r0.x, dyb = py0 - r0.y;
    if constexpr (AA) {
      const float ax = r0.z, ay = r0.w, isx = r1.x, isy = r1.y, a0 = r1.z;
      const float sx = fast_rcp(isx), sy = fast_rcp(isy);
      constexpr float tau = 6.283185307179586f;
      float g[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int i = 0; i < NSUB; ++i) {
        if ((bm[i] >> jl) & 1u) {  // warp-uniform: this sub-block can be reached at all
          const float dx = (i & 1) ? dxb + 8.f : dxb, dy = (i >> 1) ? dyb + 4.f * (i >> 1) : dyb;
          const float tx = fmaf(dy, ay, dx * ax), ty = fmaf(dy, ax, -dx * ay);
          const float zx1 = (tx + 0.5f) * isx, zx2 = (tx - 0.5f) * isx, zy1 = (ty + 0.5f) * isy, zy2 = (ty - 0.5f) * isy;
          float dx1, dx2, dy1, dy2;   // dS/dz of the four edge terms
          const float Sx = aa_sig_grad(zx1, dx1) - aa_sig_grad(zx2, dx2);
          const float Sy = aa_sig_grad(zy1, dy1) - aa_sig_grad(zy2, dy2);
          const float ix = sx * Sx, iy = sy * Sy;
          const float pa = tau * ix * iy;
          const float araw = a0 * pa;
          if (araw > thr && W[i] < sat) {
            const float alpha = fminf(araw, cmax);
            const float Ti = 1.f - W[i];
            const float w = alpha * Ti;
            W[i] += w;
            const float rinv = fast_rcp(1.f - alpha);
            float fG = 0.f;
#pragma unroll
            for (int c = 0; c < F; ++c) {
              fG = fmaf(f[c], Gd[i][c], fG);
              gf[c] = fmaf(w, Gd[i][c], gf[c]);
            }
            if constexpr (WGT) fG += Gw[i];
            RG[i] = fmaf(-fG, w, RG[i]);
            const float ag = fmaf(fG, Ti, -RG[i] * rinv);   // dL/dalpha
            const float aag = a0 * ag * tau;
            // d pdf_aa / d(mean, axis, sigma) (taichi_lib/generic.py:355-404): dS/dx = dS/dz / sigma, dS/dsigma = -z dS/dx
            const float dSx = iy * (dx1 - dx2);            // iy sx (dSx1 - dSx2) / sx
            const float dSy = ix * (dy1 - dy2);
            const float gmx = aag * fmaf(dSy, ay, -dSx * ax), gmy = -aag * fmaf(dSx, ay, dSy * ax);
            g[0] += gmx; g[1] += gmy;
            g[2] = fmaf(aag, fmaf(dSx, dx, dSy * dy), g[2]);
            g[3] = fmaf(aag, fmaf(dSx, dy, -dSy * dx), g[3]);
            g[4] = fmaf(aag * iy, Sx - fmaf(zx1, dx1, -zx2 * dx2), g[4]);
            g[5] = fmaf(aag * ix, Sy - fmaf(zy1, dy1, -zy2 * dy2), g[5]);
            g[6] = fmaf(pa, ag, g[6]);
            if (HEUR) {
              const float q = a0 * ag;
              h0 = fmaf(q, q, h0);
              h1 += fabsf(gmx) + fabsf(gmy);
            }
          }
        }
      }
#pragma unroll
      for (int k = 0; k < 7; ++k) v[k] = g[k];
    } else {
      const float a1x = r0.z, a1y = r0.w, a2x = r1.x, a2y = r1.y, l2a = r1.z;
      float M0 = 0.f, Mu = 0.f, Mw = 0.f, Muu = 0.f, Mww = 0.f, Muw = 0.f;
      const float a0h = HEUR ? fast_ex2(l2a) : 0.f;   // alpha0, once per gaussian (was one MUFU per hit)
#pragma unroll
      for (int i = 0; i < NSUB; ++i) {
        if ((bm[i] >> jl) & 1u) {  // warp-uniform: this sub-block can be reached at all
          const float dx = (i & 1) ? dxb + 8.f : dxb, dy = (i >> 1) ? dyb + 4.f * (i >> 1) : dyb;   // no x + 0.f
          const float tx = fmaf(dy, a1y, dx * a1x), ty = fmaf(dy, a2y, dx * a2x);   // k x offset / sigma, own frame
          const float araw = fast_ex2(fmaf(-ty, ty, fmaf(-tx, tx, l2a)));   // alpha0 p, as the forward forms it
          if (araw > thr && W[i] < sat) {
            const float alpha = fminf(araw, cmax);
            const float Ti = 1.f - W[i];
            const float w = alpha * Ti;
            W[i] += w;
            const float rinv = fast_rcp(1.f - alpha);
            float fG = 0.f;
#pragma unroll
            for (int c = 0; c < F; ++c) {
              fG = fmaf(f[c], Gd[i][c], fG);
              gf[c] = fmaf(w, Gd[i][c], gf[c]);
            }
            if constexpr (WGT) fG += Gw[i];
            RG[i] = fmaf(-fG, w, RG[i]);
            const float ag = fmaf(fG, Ti, -RG[i] * rinv);   // dL/dalpha
            const float gp = ag * araw;                     // alpha0 x the dL/dalpha0 share of this pixel
            const float gu = gp * tx, gw = gp * ty;
            M0 += gp; Mu += gu; Mw += gw;
            Muu = fmaf(gu, tx, Muu); Mww = fmaf(gw, ty, Mww); Muw = fmaf(gu, ty, Muw);
            if (HEUR) {
              const float aag = a0h * ag;
              h0 = fmaf(aag, aag, h0);   // |d/dmean| of this pixel: g (tx a1 + ty a2) / k^2 (the 1 / k^2 once, below)
              h1 += fabsf(fmaf(gu, a1x, gw * a2x)) + fabsf(fmaf(gu, a1y, gw * a2y));
            }
          }
        }
      }
      v[0] = M0; v[1] = Mu; v[2] = Mw; v[3] = Muu; v[4] = Mww; v[5] = Muw;
    }
#pragma unroll
    for (int c = 0; c < F; ++c) v[NM + c] = gf[c];
    if (HEUR) { v[NM + F] = h0; v[NM + F + 1] = AA ? h1 : h1 * (1.f / kHalfLog2e); }
    return (unsigned)__float_as_int(r1.w);
  };

  auto lane_done = [&]() {
    bool d = true;
#pragma unroll
    for (int i = 0; i < NSUB; ++i) d = d && (W[i] >= sat);
    return d;
  };

  // PAIR: the first survivor of a pair waits here (warp-uniform state) until the second one has been evaluated
  float held[PAIR ? NV : 1];
  unsigned held_idx = 0;
  bool holding = false;

  bool warp_done = __all_sync(kFull, lane_done());
  if (nb > 0) issue_load(0);
  for (int b = 0; b < nb; ++b) {
    const int buf = b & 1;
    if (b + 1 < nb) {
      issue_load(b + 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncwarp();
    const int n_in = min(kBwdBatch, C - b * kBwdBatch);
    if (!warp_done) {
      for (int c0 = 0; c0 < n_in; c0 += 32) {
        const int e = c0 + lane;
        // cull: bit (warp NSUB + i) of the entry's byte = it can reach sub-block i of this warp's region
        unsigned bm[NSUB];
        {
          const unsigned m = e < n_in ? (unsigned)s_mask[buf][e] >> (warp * NSUB) : 0u;
#pragma unroll
          for (int i = 0; i < NSUB; ++i) bm[i] = __ballot_sync(kFull, (m >> i) & 1u);
        }
        unsigned any = 0;
#pragma unroll
        for (int i = 0; i < NSUB; ++i) any |= bm[i];
        // the cull is tight (a survivor without a single hit is a fraction of a percent), so every survivor is
        // reduced: no vote, a miss adds zeros
        while (any) {
          const int jl = __ffs(any) - 1;
          any &= any - 1;
          const float4* ent = s_e[buf][c0 + jl];
          if constexpr (!PAIR) {
            float v[NV];
            const unsigned idx = evaluate(ent, bm, jl, v);
            reduce_scatter_step<NV, 16>(v, lane);
            if (own_base != nullptr) atomicAdd(own_base + idx * own_stride, v[0]);
          } else if (!holding) {
            held_idx = evaluate(ent, bm, jl, held);
            holding = true;
          } else {
            float v[2 * NV];
#pragma unroll
            for (int k = 0; k < NV; ++k) v[k] = held[k];
            const unsigned idx = evaluate(ent, bm, jl, v + NV);
            reduce_scatter_step<2 * NV, 16>(v, lane);
            if (pair_base != nullptr) atomicAdd(pair_base + (pair_second ? idx : held_idx) * pair_stride, v[0]);
            holding = false;
          }
        }
      }
      warp_done = __all_sync(kFull, lane_done());
    }
    __syncwarp();   // the buffer this iteration read is the one the next issue_load overwrites
    if (warp_done) break;
  }
  cp_async_wait<0>();
  if constexpr (PAIR) {
    if (holding) {   // an odd survivor is left: reduce it alone
      reduce_scatter_step<NV, 16>(held, lane);
      if (own_base != nullptr) atomicAdd(own_base + held_idx * own_stride, held[0]);
    }
  }
}

// Moments -> gradient of the packed gaussian, in place in grad_gaussians (rows hold {M0, Mt, Ms, Mtt, Mss, Mts, 0}).
// The pixel loop works in the forward record's frame: t = k u / sx, s = k w / sy with u, w the offset along / across
// the unit axis (c, s_) and k = sqrt(log2(e) / 2), and sums g = alpha0 dL/dalpha p (what ex2 returns there, times
// dL/dalpha).  Regrouping the sums of rasterizer/backward.py:170-200:
//   d/dmean  = R (Mt / (k sx), Ms / (k sy)),   d/dsigma = (Mtt / (k^2 sx), Mss / (k^2 sy)),
//   d/daxis  = (-(c P + s_ Q), c Q - s_ P) with P = (Mtt + Mss) / k^2, Q = (sx / sy - sy / sx) Mts / k^2,
//   d/dalpha0 = M0 / alpha0.
__global__ void __launch_bounds__(256)
raster_bwd_moments_kernel(int64_t V, const float* __restrict__ g2d, float* __restrict__ grad_pts) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= V) return;
  float* m = grad_pts + 7 * i;
  const float* g = g2d + 7 * i;
  const float M0 = m[0], Mt = m[1], Ms = m[2], Mtt = m[3], Mss = m[4], Mts = m[5];
  // a gaussian no pixel accumulated into keeps its zero row: rows with alpha == 0 or sigma == 0 (padding, inactive
  // points handed to rasterize() directly) would otherwise turn 0 / 0 and 0 * inf into NaN
  if (M0 == 0.f && Mt == 0.f && Ms == 0.f && Mtt == 0.f && Mss == 0.f && Mts == 0.f) return;
  const float c = g[2], s = g[3], sx = g[4], sy = g[5], a0 = g[6];
  const float isx = 1.0f / sx, isy = 1.0f / sy;
  constexpr float ik = 1.f / kSqrtHalfLog2e, ik2 = 1.f / kHalfLog2e;
  const float U = ik * isx * Mt, Vv = ik * isy * Ms;
  const float P = ik2 * (Mtt + Mss), Q = ik2 * (sx * isy - sy * isx) * Mts;
  m[0] = fmaf(c, U, -s * Vv);
  m[1] = fmaf(s, U, c * Vv);
  m[2] = -fmaf(c, P, s * Q);
  m[3] = fmaf(c, Q, -s * P);
  m[4] = ik2 * isx * Mtt;
  m[5] = ik2 * isy * Mss;
  m[6] = M0 / a0;
}

template <int F, int FP>
static int launch_bwd_fast(const GsRasterParams& p, const RasterArgs& a, const float4* rec, const float* featP,
                           cudaStream_t st) {
  const int tiles = tiles_wide(p) * tiles_high(p);
  const bool heur = p.compute_point_heuristic && a.point_heuristic != nullptr;
  const unsigned char* cmask = (const unsigned char*)a.workspace + fast_layout(p).off_mask;
  const float3 kf = make_float3((float)p.alpha_threshold, (float)p.clamp_max_alpha, (float)p.saturate_threshold);
  const float* wimg = (const float*)a.image_weight;
  const float* gw = (const float*)a.grad_image_weight;
  // Survivors are reduced in pairs (1.352 against 1.381 ms on the bench workload), except with antialiasing or the
  // weight gradient: there the paired kernel spills 84 B (F = 3) to 296 B (F = 7, heuristics) under its 64-register cap
  // and measured slower (B200, bench scene: F = 3 1.39 ms paired, 1.37 single; F = 7 2.60 / 1.84 ms;
  // benchmarks/weight_gradient.py).
#define GS_BWD_LAUNCH(HEURV, AAV, WGTV)                                                                                  \
  GS_CUDA(launch_background(raster_bwd_fast_kernel<F, FP, HEURV, !(AAV || WGTV), AAV, WGTV>, dim3(tiles * 2), dim3(32), \
                            0, st, p, rec, featP, a.tile_ranges, a.overlap_to_point, (const float*)a.image_in,       \
                            (const float*)a.grad_image, (float*)a.grad_gaussians, (float*)a.grad_features,           \
                            heur ? (float*)a.point_heuristic : nullptr, cmask, kf, wimg, gw))
#define GS_BWD_HEUR(AAV, WGTV) \
  do { if (heur) GS_BWD_LAUNCH(true, AAV, WGTV); else GS_BWD_LAUNCH(false, AAV, WGTV); } while (0)
  if (gw != nullptr) { if (p.antialias) GS_BWD_HEUR(true, true); else GS_BWD_HEUR(false, true); }
  else if (p.antialias) GS_BWD_HEUR(true, false);
  else GS_BWD_HEUR(false, false);
#undef GS_BWD_HEUR
#undef GS_BWD_LAUNCH
  GS_LAUNCH_CHECK();
  if (!p.antialias && p.points_requires_grad && a.grad_gaussians != nullptr && p.num_points > 0) {
    raster_bwd_moments_kernel<<<(unsigned)ceil_div(p.num_points, 256), 256, 0, st>>>(
        p.num_points, (const float*)a.gaussians2d, (float*)a.grad_gaussians);
    GS_LAUNCH_CHECK();
  }
  return GS_OK;
}

int raster_bwd_fast(const GsRasterParams& p, const RasterArgs& a, cudaStream_t st) {
  if (!p.workspace_holds_packed) {  // otherwise gs_raster_fwd (called with the requires_grad flags) left both there
    int rc = raster_fast_pack(p, a, /*forward=*/false, /*features=*/true, st);
    if (rc != GS_OK) return rc;
    if (p.num_features <= 7) {   // the narrow kernel reads the cull masks the forward would have left
      rc = raster_cull_mask(p, a, st);
      if (rc != GS_OK) return rc;
    }
  }
  const FastLayout L = fast_layout(p);
  unsigned char* ws = (unsigned char*)a.workspace;
  const void* featP = fast_feature_rows(p, a);
  if (p.num_features > 7)   // 8..256 channels: one pixel per lane, its own records
    return raster_bwd_wide(p, a, (const float4*)(ws + L.off_recB), featP, st);
  const float4* rec = (const float4*)(ws + (p.antialias ? L.off_recB : L.off_recF));   // the forward's records
  switch (p.num_features) {
    case 1: return launch_bwd_fast<1, 4>(p, a, rec, (const float*)featP, st);
    case 2: return launch_bwd_fast<2, 4>(p, a, rec, (const float*)featP, st);
    case 3: return launch_bwd_fast<3, 4>(p, a, rec, (const float*)featP, st);
    case 4: return launch_bwd_fast<4, 4>(p, a, rec, (const float*)featP, st);
    case 5: return launch_bwd_fast<5, 8>(p, a, rec, (const float*)featP, st);
    case 6: return launch_bwd_fast<6, 8>(p, a, rec, (const float*)featP, st);
    case 7: return launch_bwd_fast<7, 8>(p, a, rec, (const float*)featP, st);
    default: break;
  }
  GS_UNSUPPORTED("rasterizer backward (fast): %d feature channels", p.num_features);
}

}  // namespace gs
