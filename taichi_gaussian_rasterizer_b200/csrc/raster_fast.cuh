// raster_fast.cuh — shared pieces of the fast (f32, alpha blending, tile 16) rasterizer kernels:
// packed per-gaussian records, cp.async staging, the lane-parallel ellipse / pixel-block cull test.
#pragma once

#include <cuda_bf16.h>

#include <type_traits>

#include "raster.cuh"

namespace gs {

constexpr int kFastTile = 16;
constexpr int kFastTileArea = kFastTile * kFastTile;

// padded feature row length used by the fast kernels for a given F (0 = unsupported)
inline int fast_feature_pad(int F) { return F <= 4 ? 4 : F <= 8 ? 8 : F <= 16 ? 16 : F <= 36 ? 36 : F <= 64 ? 64 : 0; }
// bfloat16 feature rows (GS_BF16, 8..64 channels): a multiple of 8 channels, so that a row is whole 16 B cp.async chunks
inline int bf16_feature_pad(int F) { return F <= 8 ? 8 : F <= 16 ? 16 : F <= 40 ? 40 : F <= 64 ? 64 : 0; }

// Extra-wide features (65..256 channels): rows of xwide_row(F) floats, 64-channel slices.
constexpr int kXwideSlice = 64;
constexpr int kXwideMaxFeatures = 256;
inline bool xwide_features(int F) { return F > 64 && F <= kXwideMaxFeatures; }
__host__ __device__ inline int xwide_row(int F) { return (F + kXwideSlice - 1) / kXwideSlice * kXwideSlice; }

// Workspace layout (all 256 B aligned):
//   recF  V x 2 float4 : {mx, my, a1x, a1y} {a2x, a2y, log2(alpha), idx}       (forward records)
//   featP V x FP         : features padded to FP, f32 or bf16 like the caller's (extra-wide: empty when F is a
//                         multiple of 64, bf16: empty when F == FP; the kernels then read the caller's features in place)
//   mask  K bytes        : per tile-list entry, which of the tile's eight 8x4 pixel blocks it can reach
//   recB  V x 2 float4 : {mx, my, ax, ay} {1/sx, 1/sy, alpha, idx}             (records of the wide backward, F > 7;
//                                                                               the narrow one walks recF)
struct FastLayout {
  size_t off_recF, off_feat, off_recB, off_mask, total;
  int FP;
  bool feat_in_place;
  int feat_bytes;   // 4 (GS_F32) or 2 (GS_BF16)
};

inline FastLayout fast_layout(const GsRasterParams& p) {
  FastLayout L;
  const bool xw = xwide_features(p.num_features), bf = p.dtype == GS_BF16;
  L.FP = xw ? xwide_row(p.num_features) : bf ? bf16_feature_pad(p.num_features) : fast_feature_pad(p.num_features);
  L.feat_in_place = (xw || bf) && L.FP == p.num_features;
  L.feat_bytes = bf ? 2 : 4;
  const size_t V = (size_t)(p.num_points > 0 ? p.num_points : 1);
  size_t off = 0;
  L.off_recF = off; off += align_up(V * 32, 256);
  L.off_feat = off; off += L.feat_in_place ? 0 : align_up(V * (size_t)L.FP * L.feat_bytes, 256);
  L.off_recB = off; off += align_up(V * 32, 256);
  // one byte per tile-list entry: bit w = the entry can reach the 8x4 pixel block w of its tile (raster_cull_mask)
  L.off_mask = off; off += align_up((size_t)(p.num_overlaps > 0 ? p.num_overlaps : 1), 256);
  L.total = off;
  return L;
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ float fast_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Logistic approximation of the normal CDF used by the antialiased pdf (taichi_lib/generic.py:340-352 S_sig):
// 1 / (1 + exp(-1.6 z - 0.07 z^3)).  aa_sig_grad also returns d/dz.  The pixel integral is a DIFFERENCE of two such
// terms (cancellation: 0.04 .. 0.3 of their size), so the 2 ulp of ex2.approx / rcp.approx the plain gaussian path
// lives with would leave the image 1.2e-5 from the oracle (measured); expf and the IEEE reciprocal bring it to 4e-6.
__device__ __forceinline__ float aa_sig(float z) {
  return __frcp_rn(1.f + expf(-z * fmaf(0.07f, z * z, 1.6f)));
}
__device__ __forceinline__ float aa_sig_grad(float z, float& ds_dz) {
  const float s = aa_sig(z);
  ds_dz = fmaf(0.21f, z * z, 1.6f) * s * (1.f - s);
  return s;
}

// exp(-0.5 (tx^2 + ty^2)) == exp2(-(c tx)^2 - (c ty)^2) with c = sqrt(0.5 log2(e))
constexpr float kSqrtHalfLog2e = 0.8493218002880191f;
constexpr float kHalfLog2e = 0.7213475204444817f;

// Conservative test: can gaussian (conic A of the scaled axes, exponent budget qmax) reach any pixel centre
// of the block [x0, x1] x [y0, y1]?  Minimises the quadratic form over the rectangle exactly (interior, or the
// clamped 1-D minimum on each edge facing the mean) and adds slack for rounding; the per pixel test stays exact.
__device__ __forceinline__ bool block_may_touch(float mx, float my, float a1x, float a1y, float a2x, float a2y,
                                                float qmax, float x0, float x1, float y0, float y1) {
  const float dx0 = x0 - mx, dx1 = x1 - mx, dy0 = y0 - my, dy1 = y1 - my;
  const float dxc = fminf(fmaxf(0.f, dx0), dx1);
  const float dyc = fminf(fmaxf(0.f, dy0), dy1);
  const float A00 = a1x * a1x + a2x * a2x, A01 = a1x * a1y + a2x * a2y, A11 = a1y * a1y + a2y * a2y;
  const float dyv = fminf(fmaxf(-A01 * dxc * fast_rcp(A11), dy0), dy1);
  const float qv = A00 * dxc * dxc + 2.f * A01 * dxc * dyv + A11 * dyv * dyv;
  const float dxh = fminf(fmaxf(-A01 * dyc * fast_rcp(A00), dx0), dx1);
  const float qh = A00 * dxh * dxh + 2.f * A01 * dxh * dyc + A11 * dyc * dyc;
  return fminf(qv, qh) < qmax * 1.001f + 1e-3f;
}

// ------------------------------------------------------------------------------------------------ feature storage
// The fast kernels take the feature storage type TF as a template parameter: float (GS_F32) or __nv_bfloat16
// (GS_BF16: features, image and image gradient stored in bf16; every blend and gradient is formed in f32 registers).
template <typename TF>
constexpr bool kBf16Storage = std::is_same_v<TF, __nv_bfloat16>;
// elements of TF per 16 B cp.async chunk
template <typename TF>
constexpr int kChunkElems = 16 / (int)sizeof(TF);

__device__ __forceinline__ float to_f32(float x) { return x; }
__device__ __forceinline__ float to_f32(__nv_bfloat16 x) { return __bfloat162float(x); }
template <typename TF>
__device__ __forceinline__ TF from_f32(float x) {   // bf16: round to nearest even, once, at the end
  if constexpr (kBf16Storage<TF>) return __float2bfloat16_rn(x);
  else return x;
}
// the two bf16 values of a 32 bit word as floats (exact): element 2k sits in the low half
__device__ __forceinline__ float bf16_lo(unsigned w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16_hi(unsigned w) { return __uint_as_float(w & 0xffff0000u); }

// ------------------------------------------------------------------------------------------------ tensor cores
// D += A . B on one m16n8k8 tile, tf32 inputs, f32 accumulate (used by the wide backward kernels)
__device__ __forceinline__ void mma_tf32_16x8x8(float (&c)[4], const unsigned (&a)[4], unsigned b0, unsigned b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// x = hi + lo, both rounded to nearest tf32: residual 2^-24 |x|
__device__ __forceinline__ unsigned tf32_rna(float x) {
  unsigned r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}

// ------------------------------------------------------------------------------------------------ warp reductions
// Transposed butterfly over NV per-lane partial sums: every exchange step halves the number of live values
// (the lane keeps the half selected by its lane bit and adds the partner's copy of it), so NV values cost about
// NV shuffles instead of 5 NV.  reduce_owner<NV>(lane) tells which value ends up, fully summed, in v[0] of a lane.
template <int N, int OFF>
__device__ __forceinline__ void reduce_scatter_step(float* v, int lane) {
  if constexpr (OFF >= 1) {
    if constexpr (N > 1) {
      constexpr int H = (N + 1) / 2;
      const bool upper = (lane & OFF) != 0;
#pragma unroll
      for (int i = 0; i < H; ++i) {
        if (i + H < N) {
          const float send = upper ? v[i] : v[i + H];
          const float keep = upper ? v[i + H] : v[i];
          v[i] = keep + __shfl_xor_sync(kFull, send, OFF);
        } else {
          // odd N: the unpaired value is summed on both sides (no selects); the upper half's copy is a duplicate
          // that reduce_owner never hands out
          v[i] += __shfl_xor_sync(kFull, v[i], OFF);
        }
      }
      reduce_scatter_step<H, OFF / 2>(v, lane);
    } else {
      v[0] += __shfl_xor_sync(kFull, v[0], OFF);
      reduce_scatter_step<1, OFF / 2>(v, lane);
    }
  }
}

template <int NV>
__device__ __forceinline__ int reduce_owner(int lane) {
  int base = 0, cnt = NV, n = NV;
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    if (n > 1) {
      const int half = (n + 1) / 2;
      if (lane & off) { base += half; cnt = max(cnt - half, 0); }
      else cnt = min(cnt, half);
      n = half;
    } else if (lane & off) {
      cnt = 0;
    }
  }
  return cnt == 1 ? base : -1;
}

// the padded feature rows the fast kernels stage from (workspace, or the caller's features read in place)
inline const void* fast_feature_rows(const GsRasterParams& p, const RasterArgs& a) {
  const FastLayout L = fast_layout(p);
  return L.feat_in_place ? a.features : (const void*)((unsigned char*)a.workspace + L.off_feat);
}

int raster_fast_pack(const GsRasterParams& p, const RasterArgs& a, bool forward, bool features, cudaStream_t st);
// cull masks of every tile-list entry against the eight 8x4 pixel blocks of its tile (needs the forward records)
int raster_cull_mask(const GsRasterParams& p, const RasterArgs& a, cudaStream_t st);

// raster_fast_bwd_wide.cu: backward for 8..256 feature channels (one pixel per lane, tensor-core feature gradient)
int raster_bwd_wide(const GsRasterParams& p, const RasterArgs& a, const float4* rec, const void* featP, cudaStream_t st);

}  // namespace gs
