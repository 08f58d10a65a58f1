// raster_fast_bwd_wide.cu — backward rasterizer for WIDE feature vectors (8..256 channels; f32, alpha blending,
// tile 16), e.g. BASELINE.json's feature-lifting configuration (depth + depth^2 + 32 features = 34 channels) and
// feature fields for semantic or foundation-model distillation (128, 256 dimensions), each in one pass.
//
// Same arithmetic contract as raster_fast_bwd.cu (rasterizer/backward.py:52-228 of the reference).  With F
// channels the per pixel state of the narrow kernel (4 pixels per lane) no longer fits in registers, so the
// mapping is the forward kernel's: a warp owns an 8x4 block of a 16x16 tile, a lane ONE pixel.
//   * per pixel state: W, RG = sum_c R_c G_c and the pixel's image gradient G; the replay needs the remaining
//     features only through R . G (see raster_fast_bwd.cu),
//         alpha_grad = T (G . f_i) - RG / (1 - alpha),   RG -= w (G . f_i),
//     so R itself is never materialised — the reference keeps 2 x 4 x F floats per thread (backward.py:43-44,101-102);
//   * tile lists staged through shared memory with cp.async double buffering (records + padded feature rows, the
//     16 B chunks spread over the whole CTA); lane-parallel ellipse / block cull per warp;
//   * the 7 (+2) geometry sums of a survivor are reduced with a transposed butterfly and committed by the owning lanes
//     with red.global.add;
//   * a lane is hit at most once per gaussian, so the feature gradient of a survivor over the warp's 32 pixels is the
//     vector-matrix product d/df[c] = sum_p w[p] G[p][c].  A warp collects its survivors in groups of 16 and forms
//       D[16 survivors x F] = Wt[16 x 32 pixels] . G[32 pixels x F]
//     on the tensor cores (mma.sync m16n8k8, tf32 inputs, f32 accumulate): the lanes park their blend weights in a
//     per-warp shared-memory tile during the replay (one 8 B store per survivor), G sits in a per-warp shared-memory
//     tile for the whole tile list.  Warp butterflies spent ~4 instructions per channel and survivor on it (~150 of
//     the ~300 instructions per survivor at F = 34): 8.0 ms at config 4, 6.8 ms with the product.
//     tf32 alone (11 bit significands) would leave ~2e-4 relative error, above the 1e-4 gradient tolerance, so both
//     operands are split x = hi + lo (both rounded to nearest tf32, residual 2^-24) and three products are accumulated
//     (hi hi + lo hi + hi lo; the dropped lo lo term is 2^-22): measured error against the oracle as for the f32 path.
// Why mma.sync and not tcgen05: the product is per WARP (its own 16 survivors, its own 32 pixels), 16 x 32 x F, issued
// from inside a SIMT replay loop whose A operand is produced by the lanes a few instructions earlier; a CTA-level
// tcgen05 tile (M >= 64, operands in descriptor-addressed shared memory, accumulator in TMEM behind an mbarrier) would
// need a block-diagonal [gaussians x 256 pixels] operand of mostly zeros and two extra copies for the split.  The tensor
// work is ~1 % of the kernel's issue slots either way; what it removes is the shuffle work.
// Why G . f_i stays on the SIMT pipes: it is needed only for the lanes a survivor hits, inside the sequential replay,
// and costs F / 4 LDS.128 + F FFMA per hit lane; as a [candidates x F] . [F x 32 pixels] product it would be formed
// for every staged candidate that passes the block cull, hit or not, and the split would triple it.  Not measured.
//
// Two modes of one kernel template:
//   * FP = 8, 16, 36, 64 (F <= 64, FP = fast_feature_pad(F)): G also lives in registers for the dot product, batches of
//     32 staged entries, every channel loop fully unrolled;
//   * FP = 0, extra-wide (65..256 channels, rows of xwide_row(F) floats): G (up to 256 floats) no longer fits in
//     registers and is read from the warp's shared tile only; batches of 16 entries so that at F = 256 two CTAs of two
//     warps fit an SM (2 x 107 KB of shared memory: 32 px x 256 ch x 4 B = 32 KB of G per warp is what limits that).
// bf16 storage (GS_BF16, TF = __nv_bfloat16): image, image gradient and staged feature rows are bf16 (rows of
// bf16_feature_pad(F) or xwide_row(F) channels), every sum is formed in f32 and grad_features stays f32 (atomics).  A
// bf16 value is exact in tf32 (8 significand bits of 11), so the product needs only the weight split: W_hi G + W_lo G,
// two products instead of three, the same 2^-24 residual on W.  The extra-wide mode keeps its G tile in bf16 (half the
// shared memory: 60 instead of 110 KB per CTA at F = 256, room for three CTAs per SM instead of two); the F <= 64 modes keep the
// f32 G tile of the f32 kernel, whose B-fragment loads are conflict free and whose shared memory is not what bounds
// their occupancy (their register copy of G is f32 either way).
// The forward of the extra-wide mode is raster_fwd_fast_kernel<64, ..., XW = true> (raster_fast_fwd.cu): one CTA per
// tile and 64-channel slice.  The backward cannot be sliced that way: aag = alpha_0 * alpha_grad enters the heuristics
// as aag^2 and |pgx| + |pgy|, which are not linear in the channels, and alpha_grad itself needs the full G . f_i.
#include "raster_fast.cuh"

namespace gs {

// Two warps per CTA, four CTAs per tile, each staging the tile list for itself: the block barrier of a batch then waits
// for two warps instead of eight (21 % of the stall samples sat there).  Measured at config 4 (34 channels, 4K): eight
// warps 7.05 ms, four 7.35, two 6.39, one 6.99.
constexpr int kWideWarps = 2;
constexpr int kWideGroup = 16;   // survivors per tensor-core product (M of the mma)
constexpr int kWideWS = 36;      // row stride of the weight tile (float2 units): conflict-free A loads

// Shared memory of a CTA: two staged batches {records, feature rows}, then per warp the G tile [32][GS], the weight tile
// [16][kWideWS] of {hi, lo} and the survivors' indices [16].
// TF: feature storage; GT: element of the G tile (bf16 only in the extra-wide bf16 mode).
template <int FP, typename TF = float>
struct WideLayout {
  // staged tile-list entries per buffer (F <= 64: 64 gave 8.6 ms instead of 6.9 at config 4, the warps of a CTA drift
  // further apart between barriers)
  static constexpr int kBatch = FP > 0 ? 32 : 16;
  using GT = std::conditional_t<FP == 0, TF, float>;
  int row;   // feature row (elements of TF)
  int FP8;   // channels padded to n-tiles of 8
  // row stride of the G tile (elements of GT).  F <= 64: = 8 or 24 mod 32, so that the B-fragment loads (row = lane & 3
  // (+4), column = lane >> 2) hit 32 different banks.  Extra-wide: 16 B past a multiple of 128 B, so that a lane
  // reading its own row with LDS.128 (G . f_i) is conflict free; the f32 B fragments take two-way conflicts there (the
  // bf16 ones none: the four rows start 4 banks apart and a row's eight columns share 4 words).
  int GS;
  size_t stage_bytes, warp_bytes;
  __host__ __device__ explicit WideLayout(int F)
      : row(FP > 0 ? FP : xwide_row(F)), FP8((row + 7) / 8 * 8),
        GS(FP == 0 ? row + 16 / (int)sizeof(GT) : (FP8 % 32 == 8 || FP8 % 32 == 24) ? FP8 : FP8 + 8),
        stage_bytes((size_t)2 * kBatch * (32 + row * (int)sizeof(TF))),
        warp_bytes((size_t)32 * GS * sizeof(GT) + kWideGroup * kWideWS * 8 + kWideGroup * 4) {}
  __host__ __device__ size_t total() const { return stage_bytes + kWideWarps * warp_bytes; }
};

// WGT: the image weight W is differentiable too (gradient gw, forward W in wimg): one more channel whose feature is
// always 1, so RG starts with W_final Gw and f . G gains + Gw (see raster_bwd_fast_kernel).
template <int FP, bool HEUR, bool WGT, typename TF = float>
__global__ void __launch_bounds__(kWideWarps * 32, 8)   // eight CTAs of two warps per SM: at most 128 registers
raster_bwd_wide_mma_kernel(const __grid_constant__ GsRasterParams p, const float4* __restrict__ rec,
                           const TF* __restrict__ featP, const int32_t* __restrict__ ranges,
                           const int32_t* __restrict__ o2p, const TF* __restrict__ image,
                           const TF* __restrict__ grad_image, float* __restrict__ grad_pts,
                           float* __restrict__ grad_feat, float* __restrict__ heuristic,
                           const float* __restrict__ wimg, const float* __restrict__ gw) {
  using Layout = WideLayout<FP, TF>;
  using GT = typename Layout::GT;
  constexpr bool kBF = kBf16Storage<TF>;
  constexpr int CE = kChunkElems<TF>;   // features per 16 B chunk
  constexpr int kBatch = Layout::kBatch;
  constexpr int NG = 7 + (HEUR ? 2 : 0);             // geometry (+ heuristic) values
  constexpr int kThreads = kWideWarps * 32, kParts = 8 / kWideWarps;
  const int F = p.num_features;
  const Layout L(F);
  // literals for F <= 64 (not the layout's fields), so that the channel loops unroll fully
  const int row = FP > 0 ? FP : L.row, FP8 = FP > 0 ? (FP + 7) / 8 * 8 : L.FP8, GS = L.GS;
  extern __shared__ __align__(16) unsigned char smem[];
  float4* s_r0 = reinterpret_cast<float4*>(smem);                       // [2][kBatch]
  float4* s_r1 = s_r0 + 2 * kBatch;                                     // [2][kBatch]
  TF* s_feat = reinterpret_cast<TF*>(smem + 2 * kBatch * 32);           // [2][kBatch][row]

  const int tile = blockIdx.x / kParts, t = threadIdx.x, lane = t & 31, lwarp = t >> 5;
  const int warp = (blockIdx.x % kParts) * kWideWarps + lwarp;   // which 8x4 pixel block of the tile
  unsigned char* wbase = smem + L.stage_bytes + (size_t)lwarp * L.warp_bytes;
  GT* s_G = reinterpret_cast<GT*>(wbase);                                                        // [32][GS]
  float2* s_W = reinterpret_cast<float2*>(wbase + (size_t)32 * GS * sizeof(GT));                 // [16][WS] {hi, lo}
  int* s_idx = reinterpret_cast<int*>(wbase + (size_t)32 * GS * sizeof(GT) + kWideGroup * kWideWS * 8);   // [16]

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

  float G[FP > 0 ? FP : 1];   // F <= 64: the register copy of this lane's row of the G tile
  GT* my_G = s_G + lane * GS;
  float W = inb ? 0.f : 1.f, RG = 0.f, Gw = 0.f;
  {
    const int64_t pix = (int64_t)py * p.image_width + px;   // 64 bit: a 4K image of 256 channels has 2.1 G elements
#pragma unroll(FP > 0 ? FP : 4)
    for (int c = 0; c < row; ++c) {
      const bool ok = inb && c < F;
      const float g = ok ? to_f32(grad_image[pix * F + c]) : 0.f;
      RG = fmaf(ok ? to_f32(image[pix * F + c]) : 0.f, g, RG);
      my_G[c] = from_f32<GT>(g);   // exact: g is a value of TF
      if constexpr (FP > 0) G[c] = g;
    }
    if constexpr (WGT) {
      Gw = inb ? gw[pix] : 0.f;
      RG = fmaf(inb ? wimg[pix] : 0.f, Gw, RG);
    }
#pragma unroll
    for (int c = row; c < FP8; ++c) my_G[c] = GT();
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
        const float2 a0 = s_W[gid * kWideWS + tig + 8 * k], a1 = s_W[(gid + 8) * kWideWS + tig + 8 * k];
        const float2 a2 = s_W[gid * kWideWS + tig + 4 + 8 * k], a3 = s_W[(gid + 8) * kWideWS + tig + 4 + 8 * k];
        ahi[k][0] = __float_as_uint(a0.x); ahi[k][1] = __float_as_uint(a1.x);
        ahi[k][2] = __float_as_uint(a2.x); ahi[k][3] = __float_as_uint(a3.x);
        alo[k][0] = __float_as_uint(a0.y); alo[k][1] = __float_as_uint(a1.y);
        alo[k][2] = __float_as_uint(a2.y); alo[k][3] = __float_as_uint(a3.y);
      }
      const int s0 = gid, s1 = gid + 8;
      const int64_t i0 = s0 < ns ? s_idx[s0] : -1, i1 = s1 < ns ? s_idx[s1] : -1;
#pragma unroll(FP > 0 ? (FP + 7) / 8 : 2)
      for (int n = 0; n < FP8 / 8; ++n) {
        float c[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float b0 = to_f32(s_G[(tig + 8 * k) * GS + gid + 8 * n]);
          const float b1 = to_f32(s_G[(tig + 4 + 8 * k) * GS + gid + 8 * n]);
          if constexpr (kBF) {   // G is exact in tf32
            mma_tf32_16x8x8(c, ahi[k], __float_as_uint(b0), __float_as_uint(b1));
            mma_tf32_16x8x8(c, alo[k], __float_as_uint(b0), __float_as_uint(b1));
          } else {
            const unsigned b0h = tf32_rna(b0), b1h = tf32_rna(b1);
            const unsigned b0l = tf32_rna(b0 - __uint_as_float(b0h)), b1l = tf32_rna(b1 - __uint_as_float(b1h));
            mma_tf32_16x8x8(c, ahi[k], b0h, b1h);
            mma_tf32_16x8x8(c, alo[k], b0h, b1h);
            mma_tf32_16x8x8(c, ahi[k], b0l, b1l);
          }
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
  const int nb = (C + kBatch - 1) / kBatch;

  auto issue_load = [&](int b) {
    const int buf = b & 1;
    if (t < kBatch) {
      const int v = b * kBatch + t;
      if (v < C) {
        const int idx = o2p[start + v];
        cp_async16(&s_r0[buf * kBatch + t], rec + 2 * (int64_t)idx);
        cp_async16(&s_r1[buf * kBatch + t], rec + 2 * (int64_t)idx + 1);
      }
    }
    const int CH = row / CE;
    auto stage_chunk = [&](int q) {   // 16 B chunk q of the batch's feature rows
      const int slot = q / CH, part = q - slot * CH;
      const int v = b * kBatch + slot;
      if (v < C) {
        const int idx = o2p[start + v];
        cp_async16(s_feat + (buf * kBatch + slot) * row + part * CE, featP + (int64_t)idx * row + part * CE);
      }
    };
    if constexpr (FP > 0) {   // literal trip count, fully unrolled (rolled, the loop cost 2-3 % of the kernel time)
#pragma unroll
      for (int q0 = 0; q0 < kBatch * CH; q0 += kThreads)
        if (q0 + t < kBatch * CH) stage_chunk(q0 + t);
    } else {
      for (int q = t; q < kBatch * CH; q += kThreads) stage_chunk(q);
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
    const int n_in = min(kBatch, C - b * kBatch);
    if (!warp_done) {
      bool touch = false;
      if (lane < n_in) {
        const float4 r0 = s_r0[buf * kBatch + lane], r1 = s_r1[buf * kBatch + lane];
        const float cx = kSqrtHalfLog2e * r1.x, cy = kSqrtHalfLog2e * r1.y;
        touch = block_may_touch(r0.x, r0.y, r0.z * cx, r0.w * cx, -r0.w * cy, r0.z * cy, log2f(r1.z) - l2thr, bx0, bx1,
                                by0, by1);
      }
      unsigned mask = __ballot_sync(kFull, touch);
      while (mask) {
        const int j = __ffs(mask) - 1;
        mask &= mask - 1;
        const float4 r0 = s_r0[buf * kBatch + j], r1 = s_r1[buf * kBatch + j];
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
          // G . f_i over all channels (padded channels are zero in both)
          const TF* frow = s_feat + (buf * kBatch + j) * row;
          float fG0 = 0.f, fG1 = 0.f, fG2 = 0.f, fG3 = 0.f;   // four independent chains: the dot product is latency bound
          if constexpr (kBF) {   // eight channels per LDS.128, the chains of the f32 loop (channel c -> chain c % 4)
#pragma unroll(FP > 0 ? FP / 8 : 4)
            for (int c = 0; c < row; c += 8) {
              const uint4 f8 = *reinterpret_cast<const uint4*>(frow + c);
              float g8[8];
              if constexpr (FP > 0) {
#pragma unroll
                for (int k = 0; k < 8; ++k) g8[k] = G[c + k];
              } else {
                const uint4 u = *reinterpret_cast<const uint4*>(my_G + c);
                g8[0] = bf16_lo(u.x); g8[1] = bf16_hi(u.x); g8[2] = bf16_lo(u.y); g8[3] = bf16_hi(u.y);
                g8[4] = bf16_lo(u.z); g8[5] = bf16_hi(u.z); g8[6] = bf16_lo(u.w); g8[7] = bf16_hi(u.w);
              }
              fG0 = fmaf(bf16_lo(f8.x), g8[0], fG0); fG1 = fmaf(bf16_hi(f8.x), g8[1], fG1);
              fG2 = fmaf(bf16_lo(f8.y), g8[2], fG2); fG3 = fmaf(bf16_hi(f8.y), g8[3], fG3);
              fG0 = fmaf(bf16_lo(f8.z), g8[4], fG0); fG1 = fmaf(bf16_hi(f8.z), g8[5], fG1);
              fG2 = fmaf(bf16_lo(f8.w), g8[6], fG2); fG3 = fmaf(bf16_hi(f8.w), g8[7], fG3);
            }
          } else {
#pragma unroll(FP > 0 ? FP / 4 : 4)
            for (int c = 0; c < row; c += 4) {
              const float4 f4 = *reinterpret_cast<const float4*>(frow + c);
              float4 g4;
              if constexpr (FP > 0) g4 = make_float4(G[c], G[c + 1], G[c + 2], G[c + 3]);
              else g4 = *reinterpret_cast<const float4*>(my_G + c);
              fG0 = fmaf(f4.x, g4.x, fG0); fG1 = fmaf(f4.y, g4.y, fG1);
              fG2 = fmaf(f4.z, g4.z, fG2); fG3 = fmaf(f4.w, g4.w, fG3);
            }
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
          s_W[ns * kWideWS + lane] = make_float2(whi, __uint_as_float(tf32_rna(wl - whi)));
          if (lane == 0) s_idx[ns] = (int)idx;
          if (++ns == kWideGroup) flush_group();
        }
      }
      warp_done = __all_sync(kFull, W >= sat);
    }
    if (__syncthreads_and(warp_done)) break;
  }
  cp_async_wait<0>();
  if (ns > 0) flush_group();
}

template <int FP, bool HEUR, bool WGT, typename TF>
static int launch_wide(const GsRasterParams& p, const RasterArgs& a, const float4* rec, const void* featP,
                       cudaStream_t st) {
  const size_t smem = WideLayout<FP, TF>(p.num_features).total();
  const int tiles = tiles_wide(p) * tiles_high(p);
  // per launch: the attribute belongs to the (function, device) pair and the call costs about a microsecond
  GS_CUDA(cudaFuncSetAttribute(raster_bwd_wide_mma_kernel<FP, HEUR, WGT, TF>,
                               cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  raster_bwd_wide_mma_kernel<FP, HEUR, WGT, TF><<<tiles * (8 / kWideWarps), kWideWarps * 32, smem, st>>>(
      p, rec, (const TF*)featP, a.tile_ranges, a.overlap_to_point, (const TF*)a.image_in, (const TF*)a.grad_image,
      (float*)a.grad_gaussians, (float*)a.grad_features, HEUR ? (float*)a.point_heuristic : nullptr,
      (const float*)a.image_weight, (const float*)a.grad_image_weight);
  GS_LAUNCH_CHECK();
  return GS_OK;
}

template <int FP, typename TF = float>
static int dispatch_wide(const GsRasterParams& p, const RasterArgs& a, const float4* rec, const void* featP,
                         cudaStream_t st) {
  const bool heur = p.compute_point_heuristic && a.point_heuristic != nullptr;
  if (a.grad_image_weight != nullptr)
    return heur ? launch_wide<FP, true, true, TF>(p, a, rec, featP, st)
                : launch_wide<FP, false, true, TF>(p, a, rec, featP, st);
  return heur ? launch_wide<FP, true, false, TF>(p, a, rec, featP, st)
              : launch_wide<FP, false, false, TF>(p, a, rec, featP, st);
}

int raster_bwd_wide(const GsRasterParams& p, const RasterArgs& a, const float4* rec, const void* featP,
                    cudaStream_t st) {
  if (p.dtype == GS_BF16) {
    using bf16 = __nv_bfloat16;
    if (xwide_features(p.num_features)) return dispatch_wide<0, bf16>(p, a, rec, featP, st);
    switch (bf16_feature_pad(p.num_features)) {
      case 8: return dispatch_wide<8, bf16>(p, a, rec, featP, st);
      case 16: return dispatch_wide<16, bf16>(p, a, rec, featP, st);
      case 40: return dispatch_wide<40, bf16>(p, a, rec, featP, st);
      case 64: return dispatch_wide<64, bf16>(p, a, rec, featP, st);
      default: GS_UNSUPPORTED("rasterizer backward (wide, bf16): %d feature channels", p.num_features);
    }
  }
  if (xwide_features(p.num_features)) return dispatch_wide<0>(p, a, rec, featP, st);
  switch (fast_feature_pad(p.num_features)) {
    case 8: return dispatch_wide<8>(p, a, rec, featP, st);
    case 16: return dispatch_wide<16>(p, a, rec, featP, st);
    case 36: return dispatch_wide<36>(p, a, rec, featP, st);
    case 64: return dispatch_wide<64>(p, a, rec, featP, st);
    default: GS_UNSUPPORTED("rasterizer backward (wide): %d feature channels", p.num_features);
  }
}

}  // namespace gs
