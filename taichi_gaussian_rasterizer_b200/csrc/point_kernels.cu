// point_kernels.cu — per-gaussian kernels that are bound by HBM: spherical-harmonics forward /
// backward and the hand-derived backward of the projection.
//
// Replaces (paths relative to /root/reference/taichi_splatting/):
//   evaluate_sh_at_kernel and its Taichi-autodiff .grad      spherical_harmonics.py:118-134, :154-161
//   indexed_project_kernel.grad (Taichi autodiff)             perspective/projection.py:83-118, :164-185
// The reference obtains both backward passes from Taichi's reverse-mode autodiff; here they are
// derived by hand (DESIGN.md §projection backward) and checked against torch autograd / gradcheck.
#include "common.cuh"
#include "geom_math.cuh"

namespace gs {

// ------------------------------------------------------------------------------------------------ SH
template <typename T, int D>
__device__ __forceinline__ void sh_basis(T x, T y, T z, T* o) {
  o[0] = T(0.282094791773878);
  if (D >= 4) {
    o[1] = T(-0.48860251190292) * y;
    o[2] = T(0.48860251190292) * z;
    o[3] = T(-0.48860251190292) * x;
  }
  if (D >= 9) {
    T x2 = x * x, y2 = y * y, z2 = z * z, xy = x * y, xz = x * z, yz = y * z;
    o[4] = T(1.09254843059208) * xy;
    o[5] = T(-1.09254843059208) * yz;
    o[6] = T(0.94617469575756) * z2 - T(0.31539156525252);
    o[7] = T(-1.09254843059208) * xz;
    o[8] = T(0.54627421529604) * x2 - T(0.54627421529604) * y2;
    if (D >= 16) {
      o[9] = T(-0.590043589926644) * y * (T(3.0) * x2 - y2);
      o[10] = T(2.89061144264055) * xy * z;
      o[11] = T(0.304697199642977) * y * (T(1.5) - T(7.5) * z2);
      o[12] = T(1.24392110863372) * z * (T(1.5) * z2 - T(0.5)) - T(0.497568443453487) * z;
      o[13] = T(0.304697199642977) * x * (T(1.5) - T(7.5) * z2);
      o[14] = T(1.44530572132028) * z * (x2 - y2);
      o[15] = T(-0.590043589926644) * x * (x2 - T(3.0) * y2);
    }
  }
}

// d(basis_j)/d(x, y, z)
template <typename T, int D>
__device__ __forceinline__ void sh_basis_grad(T x, T y, T z, T* gx, T* gy, T* gz) {
  const T c1 = T(0.48860251190292), c2 = T(1.09254843059208), c3 = T(0.94617469575756),
          c5 = T(0.54627421529604), c6 = T(0.590043589926644), c7 = T(2.89061144264055),
          c8 = T(0.304697199642977), c9 = T(1.24392110863372), c10 = T(0.497568443453487),
          c11 = T(1.44530572132028);
  gx[0] = gy[0] = gz[0] = T(0);
  if (D >= 4) {
    gx[1] = T(0); gy[1] = -c1; gz[1] = T(0);
    gx[2] = T(0); gy[2] = T(0); gz[2] = c1;
    gx[3] = -c1; gy[3] = T(0); gz[3] = T(0);
  }
  if (D >= 9) {
    gx[4] = c2 * y; gy[4] = c2 * x; gz[4] = T(0);
    gx[5] = T(0); gy[5] = -c2 * z; gz[5] = -c2 * y;
    gx[6] = T(0); gy[6] = T(0); gz[6] = T(2) * c3 * z;
    gx[7] = -c2 * z; gy[7] = T(0); gz[7] = -c2 * x;
    gx[8] = T(2) * c5 * x; gy[8] = T(-2) * c5 * y; gz[8] = T(0);
    if (D >= 16) {
      T x2 = x * x, y2 = y * y, z2 = z * z;
      gx[9] = T(-6) * c6 * x * y; gy[9] = -c6 * (T(3) * x2 - T(3) * y2); gz[9] = T(0);
      gx[10] = c7 * y * z; gy[10] = c7 * x * z; gz[10] = c7 * x * y;
      gx[11] = T(0); gy[11] = c8 * (T(1.5) - T(7.5) * z2); gz[11] = T(-15) * c8 * y * z;
      gx[12] = T(0); gy[12] = T(0); gz[12] = c9 * (T(4.5) * z2 - T(0.5)) - c10;
      gx[13] = c8 * (T(1.5) - T(7.5) * z2); gy[13] = T(0); gz[13] = T(-15) * c8 * x * z;
      gx[14] = T(2) * c11 * x * z; gy[14] = T(-2) * c11 * y * z; gz[14] = c11 * (x2 - y2);
      gx[15] = -c6 * (T(3) * x2 - T(3) * y2); gy[15] = T(6) * c6 * x * y; gz[15] = T(0);
    }
  }
}

template <typename T> __device__ __forceinline__ T rsqrt_(T x);
template <> __device__ __forceinline__ float rsqrt_(float x) { return 1.0f / sqrtf(x); }
template <> __device__ __forceinline__ double rsqrt_(double x) { return 1.0 / sqrt(x); }

template <typename T, int D>
__global__ void __launch_bounds__(256)
sh_fwd_kernel(const __grid_constant__ GsSHParams p, const T* __restrict__ params, const T* __restrict__ positions,
              const int64_t* __restrict__ indexes, const T* __restrict__ cam, T* __restrict__ out,
              const int32_t* __restrict__ count_dev) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  // count_dev: number of valid indexes still on the device (gs_sh_fwd_counted); p.num_indexes is then the capacity
  const int64_t nv = count_dev ? (int64_t)*count_dev : p.num_indexes;
  if (i >= nv) return;
  const int64_t idx = indexes[i];
  const int K = p.num_channels;
  T dx = positions[3 * idx] - cam[0], dy = positions[3 * idx + 1] - cam[1], dz = positions[3 * idx + 2] - cam[2];
  T inv = rsqrt_<T>(dx * dx + dy * dy + dz * dz);
  T b[D];
  sh_basis<T, D>(dx * inv, dy * inv, dz * inv, b);
  const T* row = params + idx * K * D;
  for (int k = 0; k < K; ++k) {
    T acc = T(0);
    if (D % 4 == 0 && sizeof(T) == 4) {
      const float4* r4 = reinterpret_cast<const float4*>(row + k * D);
#pragma unroll
      for (int j = 0; j < D / 4; ++j) {
        float4 v = __ldg(r4 + j);
        acc += b[4 * j] * v.x + b[4 * j + 1] * v.y + b[4 * j + 2] * v.z + b[4 * j + 3] * v.w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < D; ++j) acc += b[j] * row[k * D + j];
    }
    T v = acc + T(0.5);
    out[i * K + k] = v < T(0) ? T(0) : (v > T(1) ? T(1) : v);
  }
}

template <typename T, int D>
__global__ void __launch_bounds__(256)
sh_bwd_kernel(const __grid_constant__ GsSHParams p, const T* __restrict__ params, const T* __restrict__ positions,
              const int64_t* __restrict__ indexes, const T* __restrict__ cam, const T* __restrict__ grad_out,
              T* __restrict__ grad_params, T* __restrict__ grad_positions, T* __restrict__ grad_cam) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int K = p.num_channels;
  T gpx = T(0), gpy = T(0), gpz = T(0);
  if (i < p.num_indexes) {
    const int64_t idx = indexes[i];
    T dx = positions[3 * idx] - cam[0], dy = positions[3 * idx + 1] - cam[1], dz = positions[3 * idx + 2] - cam[2];
    T inv = rsqrt_<T>(dx * dx + dy * dy + dz * dz);
    T x = dx * inv, y = dy * inv, z = dz * inv;
    T b[D];
    sh_basis<T, D>(x, y, z, b);
    T gb[D];  // d loss / d basis_j
#pragma unroll
    for (int j = 0; j < D; ++j) gb[j] = T(0);
    const T* row = params + idx * K * D;
    for (int k = 0; k < K; ++k) {
      T acc = T(0);
#pragma unroll
      for (int j = 0; j < D; ++j) acc += b[j] * row[k * D + j];
      T v = acc + T(0.5);
      T g = (v > T(0) && v < T(1)) ? grad_out[i * K + k] : T(0);  // clamp passes gradient strictly inside
      if (g != T(0)) {
        if (grad_params) {
          T* gr = grad_params + (idx * K + k) * D;
#pragma unroll
          for (int j = 0; j < D; ++j) red_add(gr + j, g * b[j]);
        }
#pragma unroll
        for (int j = 0; j < D; ++j) gb[j] += g * row[k * D + j];
      }
    }
    if (grad_positions || grad_cam) {
      T gx[D], gy[D], gz[D];
      sh_basis_grad<T, D>(x, y, z, gx, gy, gz);
      T ddx = T(0), ddy = T(0), ddz = T(0);  // grad wrt the unit direction
#pragma unroll
      for (int j = 0; j < D; ++j) { ddx += gb[j] * gx[j]; ddy += gb[j] * gy[j]; ddz += gb[j] * gz[j]; }
      T dot = ddx * x + ddy * y + ddz * z;  // through normalize: (I - d d^T) / |v|
      gpx = (ddx - x * dot) * inv; gpy = (ddy - y * dot) * inv; gpz = (ddz - z * dot) * inv;
      if (grad_positions) {
        red_add(grad_positions + 3 * idx, gpx);
        red_add(grad_positions + 3 * idx + 1, gpy);
        red_add(grad_positions + 3 * idx + 2, gpz);
      }
    }
  }
  if (grad_cam) {  // camera position receives minus the sum of the point gradients
    __shared__ T s_red[3][8];
    T sx = warp_sum(gpx), sy = warp_sum(gpy), sz = warp_sum(gpz);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { s_red[0][warp] = sx; s_red[1][warp] = sy; s_red[2][warp] = sz; }
    __syncthreads();
    if (threadIdx.x < 3) {
      T t = T(0);
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += s_red[threadIdx.x][w];
      if (t != T(0)) red_add(grad_cam + threadIdx.x, -t);
    }
  }
}

// Dense SH backward for the render path: `indexes` strictly ascending (the visible set that gs_project_fwd
// compacts), f32, K*D a multiple of 4.  A block owns 128 consecutive visible points AND every gaussian row
// between them: coefficient rows are staged to shared memory with coalesced 16 B loads (12 lanes per 192 B row),
// each thread turns its row into the gradient row in place, and the rows go back with coalesced 16 B stores.
// Rows of culled gaussians inside the block's span are zero-filled by the same block (FILL), so grad_params /
// grad_positions need no memset and no atomics: 2 x 4 K D bytes per gaussian of traffic in total.
constexpr int kSHDenseBlock = 128;

// FROM_OUT: `params` holds the forward OUTPUT (V, K) instead of the coefficients.  The coefficient gradient
// g_k b_j needs the coefficients only for the clamp mask, and v in (0, 1) <=> clamp(v) in (0, 1): when no position /
// camera gradient is asked for, the 4 K D byte row gather per gaussian (a third of the kernel's traffic) is skipped.
//
// A16: the gathered coefficient rows (unless FROM_OUT) and the gradient rows move in 16 B units, which needs K D a
// multiple of 4 and 16 B aligned `params` / `grad_params`.  !A16 moves them in 4 B units (4 B cp.async for the gather),
// at any alignment: rows of 3 or 27 floats (D = 1, 9) at idx * 12 B or idx * 108 B, or misaligned pointers at D = 4, 16.
// Odd row lengths sit back to back in shared memory (odd stride: conflict-free scalar LDS / STS per thread).
template <int K, int D, bool FILL, bool FROM_OUT = false, bool A16 = true>
__global__ void __launch_bounds__(kSHDenseBlock, 6)
sh_bwd_dense_kernel(const __grid_constant__ GsSHParams p, const float* __restrict__ params,
                    const float* __restrict__ positions, const int64_t* __restrict__ indexes,
                    const float* __restrict__ cam, const float* __restrict__ grad_out, float* __restrict__ grad_params,
                    float* __restrict__ grad_positions, float* __restrict__ grad_cam) {
  constexpr int RL = K * D, R4 = RL / 4, S4 = (R4 + 1) | 1;  // odd float4 stride: conflict-free LDS.128 per thread
  constexpr bool V4 = RL % 4 == 0;                            // rows of whole float4s: padded rows in shared memory
  constexpr int SR = V4 ? 4 * S4 : RL;                        // shared row stride in floats
  static_assert(V4 || !A16, "16 B row units need a row length that is a multiple of 4 floats");
  __shared__ float4 s_row[V4 ? kSHDenseBlock * S4 : (kSHDenseBlock * RL + 3) / 4];
  __shared__ int64_t s_idx[kSHDenseBlock + 1];
  __shared__ float s_red[3][kSHDenseBlock / 32];
  float* s_f = reinterpret_cast<float*>(s_row);

  const int t = threadIdx.x;
  const int64_t i0 = (int64_t)blockIdx.x * kSHDenseBlock;
  const int nrows = (int)min((int64_t)kSHDenseBlock, p.num_indexes - i0);
  const bool last_block = i0 + nrows == p.num_indexes;
  if (t < nrows) s_idx[t + 1] = indexes[i0 + t];
  if (t == 0) s_idx[0] = i0 > 0 ? indexes[i0 - 1] : -1;
  __syncthreads();

  if (!FROM_OUT) {
    if constexpr (A16) {
#pragma unroll
      for (int m = 0; m < R4; ++m) {  // R4 independent 16 B cp.async gathers in flight per thread, no staging registers
        const int q = t + m * kSHDenseBlock, r = q / R4, part = q - r * R4;
        if (q < nrows * R4) {
          const unsigned dst = (unsigned)__cvta_generic_to_shared(&s_row[r * S4 + part]);
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst),
                       "l"(reinterpret_cast<const float4*>(params + s_idx[r + 1] * RL) + part) : "memory");
        }
      }
    } else {
#pragma unroll 4
      for (int m = 0; m < RL; ++m) {  // RL 4 B cp.async gathers per thread; consecutive lanes read consecutive floats
        const int q = t + m * kSHDenseBlock, r = q / RL, part = q - r * RL;
        if (q < nrows * RL) {
          const unsigned dst = (unsigned)__cvta_generic_to_shared(&s_f[r * SR + part]);
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(params + s_idx[r + 1] * RL + part)
                       : "memory");
        }
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
  }

  float gpx = 0.f, gpy = 0.f, gpz = 0.f;
  if (t < nrows) {
    const int64_t idx = s_idx[t + 1];
    const int64_t i = i0 + t;
    const float dx = positions[3 * idx] - cam[0], dy = positions[3 * idx + 1] - cam[1],
                dz = positions[3 * idx + 2] - cam[2];
    const float inv = rsqrt_<float>(dx * dx + dy * dy + dz * dz);
    const float x = dx * inv, y = dy * inv, z = dz * inv;
    float b[D], gb[D];
    sh_basis<float, D>(x, y, z, b);
#pragma unroll
    for (int j = 0; j < D; ++j) gb[j] = 0.f;
    float4* row = s_row + t * S4;
    float* row_f = s_f + t * SR;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      float v;
      float c[D];
      if (FROM_OUT) {
        v = params[i * K + k];  // the clamped forward value: inside (0, 1) exactly when the unclamped one is
      } else {
        if constexpr (D % 4 == 0) {
#pragma unroll
          for (int j4 = 0; j4 < D / 4; ++j4) {
            const float4 q4 = row[k * (D / 4) + j4];
            c[4 * j4] = q4.x; c[4 * j4 + 1] = q4.y; c[4 * j4 + 2] = q4.z; c[4 * j4 + 3] = q4.w;
          }
        } else {
#pragma unroll
          for (int j = 0; j < D; ++j) c[j] = row_f[k * D + j];
        }
        float acc = 0.f;
#pragma unroll
        for (int j = 0; j < D; ++j) acc += b[j] * c[j];
        v = acc + 0.5f;
      }
      const float g = (v > 0.f && v < 1.f) ? grad_out[i * K + k] : 0.f;  // clamp passes gradient strictly inside
      if (!FROM_OUT) {
#pragma unroll
        for (int j = 0; j < D; ++j) gb[j] += g * c[j];
      }
      if constexpr (D % 4 == 0) {
#pragma unroll
        for (int j4 = 0; j4 < D / 4; ++j4)
          row[k * (D / 4) + j4] = make_float4(g * b[4 * j4], g * b[4 * j4 + 1], g * b[4 * j4 + 2], g * b[4 * j4 + 3]);
      } else {
#pragma unroll
        for (int j = 0; j < D; ++j) row_f[k * D + j] = g * b[j];
      }
    }
    if (!FROM_OUT && (grad_positions || grad_cam)) {
      float gx[D], gy[D], gz[D];
      sh_basis_grad<float, D>(x, y, z, gx, gy, gz);
      float ddx = 0.f, ddy = 0.f, ddz = 0.f;
#pragma unroll
      for (int j = 0; j < D; ++j) { ddx += gb[j] * gx[j]; ddy += gb[j] * gy[j]; ddz += gb[j] * gz[j]; }
      const float dot = ddx * x + ddy * y + ddz * z;
      gpx = (ddx - x * dot) * inv; gpy = (ddy - y * dot) * inv; gpz = (ddz - z * dot) * inv;
      if (grad_positions) {
        grad_positions[3 * idx] = gpx; grad_positions[3 * idx + 1] = gpy; grad_positions[3 * idx + 2] = gpz;
      }
    }
  }
  __syncthreads();

  if constexpr (A16) {
#pragma unroll
    for (int m = 0; m < R4; ++m) {
      const int q = t + m * kSHDenseBlock, r = q / R4, part = q - r * R4;
      if (q < nrows * R4) {
        float4* dst = reinterpret_cast<float4*>(grad_params + s_idx[r + 1] * RL) + part;
        *dst = s_row[r * S4 + part];
      }
    }
  } else {
#pragma unroll 4
    for (int m = 0; m < RL; ++m) {
      const int q = t + m * kSHDenseBlock, r = q / RL, part = q - r * RL;
      if (q < nrows * RL) grad_params[s_idx[r + 1] * RL + part] = s_f[r * SR + part];
    }
  }

  if (FILL) {  // zero the rows of culled gaussians in (previous visible index, this block's last index] (+ the tail)
    const bool my_gap = t < nrows && s_idx[t + 1] - s_idx[t] > 1;
    const bool tail = last_block && s_idx[nrows] + 1 < p.num_points;
    if (__syncthreads_or(my_gap) || tail) {
      const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int r = 0; r <= nrows; ++r) {
        int64_t lo, hi;
        if (r < nrows) { lo = s_idx[r] + 1; hi = s_idx[r + 1]; }
        else if (tail) { lo = s_idx[nrows] + 1; hi = p.num_points; }
        else break;
        if (hi <= lo) continue;
        if constexpr (A16) {
          float4* gp4 = reinterpret_cast<float4*>(grad_params + lo * RL);
          for (int64_t q = t; q < (hi - lo) * R4; q += kSHDenseBlock) gp4[q] = z4;
        } else {
          float* gp = grad_params + lo * RL;
          for (int64_t q = t; q < (hi - lo) * RL; q += kSHDenseBlock) gp[q] = 0.f;
        }
        if (grad_positions)
          for (int64_t q = t; q < (hi - lo) * 3; q += kSHDenseBlock) grad_positions[lo * 3 + q] = 0.f;
      }
    }
  }

  if (grad_cam) {  // camera position receives minus the sum of the point gradients
    const float sx = warp_sum(gpx), sy = warp_sum(gpy), sz = warp_sum(gpz);
    const int lane = t & 31, warp = t >> 5;
    if (lane == 0) { s_red[0][warp] = sx; s_red[1][warp] = sy; s_red[2][warp] = sz; }
    __syncthreads();
    if (t < 3) {
      float s = 0.f;
      for (int w = 0; w < kSHDenseBlock / 32; ++w) s += s_red[t][w];
      if (s != 0.f) red_add(grad_cam + t, -s);
    }
  }
}

// ------------------------------------------------------------------------------------------------ deferred SH bwd
// A multi-view batch accumulates grad_params (M, K, D) over its views; done per view that is a read-modify-write of
// the whole 4 K D byte row per gaussian and view.  The coefficient gradient of one view is the outer product of the
// masked colour gradient g (K floats) with the basis b(direction) (D floats), and b is a cheap function of the
// gaussian's position and the camera centre: so a view only STAGES g (K floats per gaussian, dense over M, zero
// where culled or clamped) and ONE flush per batch forms sum_v g_v (x) b_v in registers and adds it to the row.
// Per view 4 K (2 V + M) + 8 V bytes instead of 8 K D M; per flush 4 K M (views + 2 D) + 12 M.
template <int K>
__global__ void __launch_bounds__(256)
sh_bwd_stage_kernel(int64_t nv, const float* __restrict__ out_fwd, const int64_t* __restrict__ indexes,
                    const float* __restrict__ grad_out, float* __restrict__ staged,
                    const int32_t* __restrict__ count_dev = nullptr) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (count_dev) nv = min(nv, (int64_t)*count_dev);   // counted variant: nv is the capacity
  if (j >= nv) return;
  const int64_t idx = indexes[j];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const float v = out_fwd[j * K + k];   // clamped forward value: strictly inside (0, 1) iff the unclamped one is
    staged[idx * K + k] = (v > 0.f && v < 1.f) ? grad_out[j * K + k] : 0.f;
  }
}

constexpr int kSHMaxDeferred = 16;   // GS_SH_MAX_DEFERRED_VIEWS
struct SHFlushViews {
  const float* staged[kSHMaxDeferred];
  const float* cam[kSHMaxDeferred];
};

// OVERWRITE: grad_params = the batch's sum (the caller knows the rows hold nothing yet: no zero fill before, no read here)
// A16: grad_params is 16 B aligned and read / written in float4 units.  A block's rows are one contiguous span of
// 128 K D floats, a multiple of four at every D, so the span of every block starts 16 B aligned as well; rows of 3 or
// 27 floats (D = 1, 9) sit back to back in shared memory (odd stride: conflict-free scalar STS) and go out as the
// span's float4s plus, in the last block, a tail of at most three floats.  !A16: 4 B units, at any alignment.
template <int K, int D, bool OVERWRITE, bool A16 = true>
__global__ void __launch_bounds__(kSHDenseBlock, 4)
sh_bwd_flush_kernel(int64_t n, int num_views, const __grid_constant__ SHFlushViews views,
                    const float* __restrict__ positions, float* __restrict__ grad_params) {
  constexpr int RL = K * D, R4 = RL / 4, S4 = (R4 + 1) | 1;   // odd float4 stride: conflict-free LDS.128 / STS.128
  constexpr bool V4 = RL % 4 == 0;                             // rows of whole float4s: padded rows in shared memory
  __shared__ float4 s_row[V4 ? kSHDenseBlock * S4 : kSHDenseBlock * RL / 4];
  const int t = threadIdx.x;
  const int64_t i0 = (int64_t)blockIdx.x * kSHDenseBlock, i = i0 + t;
  const int nrows = (int)min((int64_t)kSHDenseBlock, n - i0);

  float acc[RL];
#pragma unroll
  for (int q = 0; q < RL; ++q) acc[q] = 0.f;
  if (t < nrows) {
    const float px = positions[3 * i], py = positions[3 * i + 1], pz = positions[3 * i + 2];
    for (int v = 0; v < num_views; ++v) {
      float g[K];
      bool any = false;
#pragma unroll
      for (int k = 0; k < K; ++k) { g[k] = views.staged[v][i * K + k]; any = any || g[k] != 0.f; }
      if (!any) continue;
      const float* cam = views.cam[v];
      const float dx = px - cam[0], dy = py - cam[1], dz = pz - cam[2];
      const float inv = rsqrt_<float>(dx * dx + dy * dy + dz * dz);
      float b[D];
      sh_basis<float, D>(dx * inv, dy * inv, dz * inv, b);
#pragma unroll
      for (int k = 0; k < K; ++k)
#pragma unroll
        for (int j = 0; j < D; ++j) acc[k * D + j] = fmaf(g[k], b[j], acc[k * D + j]);
    }
  }
  float* s_f = reinterpret_cast<float*>(s_row);
  if constexpr (V4) {
#pragma unroll
    for (int q4 = 0; q4 < R4; ++q4)
      s_row[t * S4 + q4] = make_float4(acc[4 * q4], acc[4 * q4 + 1], acc[4 * q4 + 2], acc[4 * q4 + 3]);
  } else {
#pragma unroll
    for (int q = 0; q < RL; ++q) s_f[t * RL + q] = acc[q];
  }
  __syncthreads();
  if constexpr (V4 && A16) {
    float4* dst = reinterpret_cast<float4*>(grad_params + i0 * RL);   // the block's rows are contiguous
#pragma unroll
    for (int m = 0; m < R4; ++m) {
      const int q = t + m * kSHDenseBlock, r = q / R4, part = q - r * R4;
      if (q < nrows * R4) {
        float4 a = s_row[r * S4 + part];
        if (!OVERWRITE) {
          const float4 o = dst[q];
          a.x += o.x; a.y += o.y; a.z += o.z; a.w += o.w;
        }
        dst[q] = a;
      }
    }
  } else if constexpr (A16) {   // odd row length: s_row holds the span as it lies in global memory
    float4* dst = reinterpret_cast<float4*>(grad_params + i0 * RL);
    const int nf = nrows * RL, n4 = nf >> 2;
#pragma unroll
    for (int m = 0; m < (RL + 3) / 4; ++m) {
      const int q = t + m * kSHDenseBlock;
      if (q < n4) {
        float4 a = s_row[q];
        if (!OVERWRITE) {
          const float4 o = dst[q];
          a.x += o.x; a.y += o.y; a.z += o.z; a.w += o.w;
        }
        dst[q] = a;
      }
    }
    if (t < nf - 4 * n4) {   // last block only: the span ends inside a float4
      const int q = 4 * n4 + t;
      grad_params[i0 * RL + q] = OVERWRITE ? s_f[q] : s_f[q] + grad_params[i0 * RL + q];
    }
  } else {
    float* dst = grad_params + i0 * RL;
#pragma unroll
    for (int m = 0; m < RL; ++m) {
      const int q = t + m * kSHDenseBlock, r = q / RL, part = q - r * RL;
      if (q < nrows * RL) {
        const float a = s_f[V4 ? r * 4 * S4 + part : q];
        dst[q] = OVERWRITE ? a : a + dst[q];
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ batched SH fwd
// The forward counterpart of the deferred gradient: the views of a batch all read the same (M, K, D) coefficients,
// 4 K D bytes per gaussian and view.  One pass holds a gaussian's row in registers and evaluates it for every view
// of the batch (dense (M, K) colours per view, 4 K bytes each); a view then only gathers its visible rows.
struct SHViewsOut {
  float* out[kSHMaxDeferred];
  const float* cam[kSHMaxDeferred];
};

// A16: the rows are read as float4 (K D a multiple of 4 and `params` 16 B aligned); else one float at a time (rows of
// 3 or 27 floats, or a misaligned `params`).  Either way the sum runs in sh_fwd_kernel's order, so the colours are
// evaluate_sh_at's.
template <int K, int D, bool A16 = true>
__global__ void __launch_bounds__(128)
sh_fwd_views_kernel(int64_t n, int num_views, const __grid_constant__ SHViewsOut views,
                    const float* __restrict__ params, const float* __restrict__ positions) {
  static_assert(!A16 || (K * D) % 4 == 0, "float4 rows need K * D to be a multiple of 4");
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float c[K * D];
  if constexpr (A16) {
    const float4* r4 = reinterpret_cast<const float4*>(params + i * K * D);
#pragma unroll
    for (int q = 0; q < K * D / 4; ++q) {
      const float4 v = __ldg(r4 + q);
      c[4 * q] = v.x; c[4 * q + 1] = v.y; c[4 * q + 2] = v.z; c[4 * q + 3] = v.w;
    }
  } else {
#pragma unroll
    for (int q = 0; q < K * D; ++q) c[q] = __ldg(params + i * K * D + q);
  }
  const float px = positions[3 * i], py = positions[3 * i + 1], pz = positions[3 * i + 2];
  for (int v = 0; v < num_views; ++v) {
    const float* cam = views.cam[v];
    const float dx = px - cam[0], dy = py - cam[1], dz = pz - cam[2];
    const float inv = rsqrt_<float>(dx * dx + dy * dy + dz * dz);
    float b[D];
    sh_basis<float, D>(dx * inv, dy * inv, dz * inv, b);
#pragma unroll
    for (int k = 0; k < K; ++k) {
      float acc = 0.f;
      if constexpr (D % 4 == 0) {   // same summation order as sh_fwd_kernel: groups of four ...
#pragma unroll
        for (int j = 0; j < D / 4; ++j)
          acc += b[4 * j] * c[k * D + 4 * j] + b[4 * j + 1] * c[k * D + 4 * j + 1] +
                 b[4 * j + 2] * c[k * D + 4 * j + 2] + b[4 * j + 3] * c[k * D + 4 * j + 3];
      } else {                      // ... or one term at a time (its scalar branch)
#pragma unroll
        for (int j = 0; j < D; ++j) acc += b[j] * c[k * D + j];
      }
      const float val = acc + 0.5f;
      views.out[v][i * K + k] = val < 0.f ? 0.f : (val > 1.f ? 1.f : val);
    }
  }
}

// out[j] = src[indexes[j]] for j < *count_dev (rows of K floats; the count is still on the device)
template <int K>
__global__ void __launch_bounds__(256)
gather_rows_counted_kernel(int64_t capacity, const float* __restrict__ src, const int64_t* __restrict__ indexes,
                           const int32_t* __restrict__ count_dev, float* __restrict__ out) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nv = count_dev ? (int64_t)*count_dev : capacity;
  if (j >= nv || j >= capacity) return;
  const int64_t idx = indexes[j];
#pragma unroll
  for (int k = 0; k < K; ++k) out[j * K + k] = src[idx * K + k];
}

// Generic row gather / scatter for the visible set (any row width, strided destination / source rows): replaces
// `features[indexes]` (ATen's vectorized_gather_kernel: 1.04 ms for 2 M rows of 32 floats) and its backward
// (index_put with accumulate: a radix sort of the indexes + 0.53 ms) in the renderer's plain-feature path
// (renderer.py:152-153 of the reference: `features = gaussians.feature[indexes]`).  One thread per float, rows
// contiguous in the dense tensor, so both sides are coalesced.  The indexes are unique (the visible set), so the
// scatter needs no atomics; the count may still be on the device.
//   gather : out[j * out_stride + out_offset + c] = src[indexes[j] * row + c]
//   scatter: dst[indexes[j] * row + c] = src[j * src_stride + src_offset + c]      (dst zero-filled by the caller)
// IdxT: uint32_t when the element count fits (a 64 bit division per thread costs more than the copy); T: float, or
// uint16_t for bf16 rows (gs_*_rows_strided_u16)
template <typename IdxT, typename T = float>
__global__ void __launch_bounds__(256)
gather_rows_strided_kernel(int64_t capacity, int row, const T* __restrict__ src, const int64_t* __restrict__ indexes,
                           const int32_t* __restrict__ count_dev, T* __restrict__ out, int out_stride,
                           int out_offset) {
  const IdxT e = (IdxT)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nv = count_dev ? min(capacity, (int64_t)*count_dev) : capacity;
  const IdxT jq = e / (IdxT)row;
  const int64_t j = (int64_t)jq;
  if (j >= nv) return;
  const int c = (int)(e - jq * (IdxT)row);
  out[j * out_stride + out_offset + c] = src[indexes[j] * row + c];
}

template <typename IdxT, typename T = float>
__global__ void __launch_bounds__(256)
scatter_rows_strided_kernel(int64_t capacity, int row, const T* __restrict__ src, int src_stride, int src_offset,
                            const int64_t* __restrict__ indexes, const int32_t* __restrict__ count_dev,
                            T* __restrict__ dst) {
  const IdxT e = (IdxT)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nv = count_dev ? min(capacity, (int64_t)*count_dev) : capacity;
  const IdxT jq = e / (IdxT)row;
  const int64_t j = (int64_t)jq;
  if (j >= nv) return;
  const int c = (int)(e - jq * (IdxT)row);
  dst[indexes[j] * row + c] = src[j * src_stride + src_offset + c];
}

// Channel split / merge of the rendered image for render_depth: (P, F) rows -> (P, S) and (P, F - S), and back.
// The reference slices (renderer.py:215-222); as strided views every later elementwise pass over the 34-channel 4K
// image and autograd's zero-padded slice backward run at a fraction of the bandwidth (ATen's generic strided copy:
// four passes of 0.5 ms at config 4).  VEC floats per thread (2 when F and S are even: all three row starts 8 B aligned).
template <int VEC, typename IdxT>
__global__ void __launch_bounds__(256)
split_channels_kernel(int64_t total, int F, int S, const float* __restrict__ src, float* __restrict__ a,
                      float* __restrict__ b) {
  const IdxT eq = ((IdxT)blockIdx.x * blockDim.x + threadIdx.x) * VEC;
  const int64_t e = (int64_t)eq;
  if (e >= total) return;
  const IdxT rq = eq / (IdxT)F;
  const int64_t row = (int64_t)rq;
  const int c = (int)(eq - rq * (IdxT)F);
  float* dst = c < S ? a + row * S + c : b + row * (F - S) + (c - S);
  if (VEC == 2) *reinterpret_cast<float2*>(dst) = *reinterpret_cast<const float2*>(src + e);
  else *dst = src[e];
}

template <int VEC, typename IdxT>
__global__ void __launch_bounds__(256)
merge_channels_kernel(int64_t total, int F, int S, const float* __restrict__ a, const float* __restrict__ b,
                      float* __restrict__ dst) {
  const IdxT eq = ((IdxT)blockIdx.x * blockDim.x + threadIdx.x) * VEC;
  const int64_t e = (int64_t)eq;
  if (e >= total) return;
  const IdxT rq = eq / (IdxT)F;
  const int64_t row = (int64_t)rq;
  const int c = (int)(eq - rq * (IdxT)F);
  const float* src = c < S ? (a ? a + row * S + c : nullptr) : (b ? b + row * (F - S) + (c - S) : nullptr);
  if (VEC == 2) *reinterpret_cast<float2*>(dst + e) = src ? *reinterpret_cast<const float2*>(src) : make_float2(0.f, 0.f);
  else dst[e] = src ? *src : 0.f;
}

// ------------------------------------------------------------------------------------------------ projection bwd
constexpr int kPBwdBlock = 128;

// ACC: add into the caller's gradient buffers (visible rows only) instead of overwriting them.
template <typename T, bool ACC>
__global__ void __launch_bounds__(kPBwdBlock, sizeof(T) == 4 ? 8 : 1)
project_bwd_kernel(const __grid_constant__ GsProjectParams p, int64_t num_visible, const T* __restrict__ position,
                   const T* __restrict__ log_scaling, const T* __restrict__ rotation,
                   const T* __restrict__ alpha_logit, const T* __restrict__ Tcw, const T* __restrict__ proj,
                   const int64_t* __restrict__ indexes, const T* __restrict__ grad_points,
                   const T* __restrict__ grad_depth, T* __restrict__ g_position, T* __restrict__ g_log_scaling,
                   T* __restrict__ g_rotation, T* __restrict__ g_alpha_logit, T* __restrict__ g_Tcw,
                   T* __restrict__ g_proj, const int32_t* __restrict__ count_dev) {
  const int64_t i = (int64_t)blockIdx.x * kPBwdBlock + threadIdx.x;
  if (count_dev) num_visible = min(num_visible, (int64_t)*count_dev);   // counted variant: the capacity was passed
  CameraConst<T> C;
#pragma unroll
  for (int k = 0; k < 12; ++k) C.Tcw[k] = Tcw[k];
  C.fx = proj[0]; C.fy = proj[1]; C.cx = proj[2]; C.cy = proj[3];
  C.w = T(p.image_width); C.h = T(p.image_height);
  C.near_ = T(p.near_plane); C.far_ = T(p.far_plane); C.blur = T(p.blur_cov);
  C.lo_x = T(-(double)p.image_width * p.clamp_margin);
  C.lo_y = T(-(double)p.image_height * p.clamp_margin);
  C.hi_x = T(((double)p.image_width - 1.0) * (1.0 + p.clamp_margin));
  C.hi_y = T(((double)p.image_height - 1.0) * (1.0 + p.clamp_margin));
  C.alpha_threshold = T(p.alpha_threshold);

  T cam_grad[16];  // dW (3x3 in rows 0..2, cols 0..2), dt (col 3), then dfx dfy dcx dcy
#pragma unroll
  for (int k = 0; k < 16; ++k) cam_grad[k] = T(0);

  if (i < num_visible) {
    const int64_t idx = indexes[i];
    T pos[3] = {position[3 * idx], position[3 * idx + 1], position[3 * idx + 2]};
    T ls[3] = {log_scaling[3 * idx], log_scaling[3 * idx + 1], log_scaling[3 * idx + 2]};
    T q[4] = {rotation[4 * idx], rotation[4 * idx + 1], rotation[4 * idx + 2], rotation[4 * idx + 3]};
    ProjectState<T> S;
    Projected<T> o = project_one<T>(pos, ls, q, alpha_logit[idx], C, &S);

    const T* gp = grad_points + 7 * i;
    const T d_mean_x = gp[0], d_mean_y = gp[1], d_axis_x = gp[2], d_axis_y = gp[3];
    const T d_sig0 = gp[4], d_sig1 = gp[5], d_alpha = gp[6];
    const T d_depth = grad_depth ? grad_depth[i] : T(0);

    // 1. alpha = sigmoid(logit)
    const T d_logit = d_alpha * o.alpha * (T(1) - o.alpha);
    // 2. sigma = sqrt(lambda), axis = n / |n|, n = (a - l2, b)
    T dl1 = d_sig0 / (T(2) * o.sigma_x);
    T dl2 = d_sig1 / (T(2) * o.sigma_y);
    T da = T(0), db = T(0), dc = T(0);
    if (S.nn > T(0)) {
      T dotv = o.axis_x * d_axis_x + o.axis_y * d_axis_y;
      T dnx = (d_axis_x - o.axis_x * dotv) / S.nn;
      T dny = (d_axis_y - o.axis_y * dotv) / S.nn;
      da += dnx; dl2 -= dnx; db += dny;
    }
    // 3. eigenvalues of [[a, b], [b, c]]
    T dtr = (dl1 + dl2) * T(0.5);
    T dsg = (dl1 - dl2) * T(0.5);
    T dgap = S.sg > T(0) ? dsg / (T(2) * S.sg) : T(0);
    T tr = S.a + S.c;
    dtr += T(2) * tr * dgap;
    T ddet = T(-4) * dgap;
    da += dtr + S.c * ddet;
    dc += dtr + S.a * ddet;
    db += T(-2) * S.b * ddet;
    // 4. cov = M M^T (upper triangle read): dM = [[2da, db], [db, 2dc]] M
    T dM[2][3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      dM[0][j] = T(2) * da * S.m[0][j] + db * S.m[1][j];
      dM[1][j] = db * S.m[0][j] + T(2) * dc * S.m[1][j];
    }
    // rebuild R, RS, J, B = W RS
    const T x = S.q[0], y = S.q[1], z = S.q[2], w = S.q[3];
    T R[3][3] = {{T(1) - T(2) * y * y - T(2) * z * z, T(2) * x * y - T(2) * w * z, T(2) * x * z + T(2) * w * y},
                 {T(2) * x * y + T(2) * w * z, T(1) - T(2) * x * x - T(2) * z * z, T(2) * y * z - T(2) * w * x},
                 {T(2) * x * z - T(2) * w * y, T(2) * y * z + T(2) * w * x, T(1) - T(2) * x * x - T(2) * y * y}};
    const T zc = S.cam[2];
    const T J00 = C.fx / zc, J02 = -(S.tu - C.cx) / zc, J11 = C.fy / zc, J12 = -(S.tv - C.cy) / zc;
    T B[3][3];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int j = 0; j < 3; ++j)
        B[r][j] = (C.Tcw[r * 4 + 0] * R[0][j] + C.Tcw[r * 4 + 1] * R[1][j] + C.Tcw[r * 4 + 2] * R[2][j]) * S.s[j];
    // 5. M = J B
    T dJ00 = T(0), dJ02 = T(0), dJ11 = T(0), dJ12 = T(0);
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      dJ00 += dM[0][j] * B[0][j]; dJ02 += dM[0][j] * B[2][j];
      dJ11 += dM[1][j] * B[1][j]; dJ12 += dM[1][j] * B[2][j];
    }
    T dB[3][3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      dB[0][j] = J00 * dM[0][j];
      dB[1][j] = J11 * dM[1][j];
      dB[2][j] = J02 * dM[0][j] + J12 * dM[1][j];
    }
    // B = W RS: dW += dB RS^T ; dRS = W^T dB
    T dRS[3][3];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        cam_grad[r * 4 + j] += dB[r][0] * R[j][0] * S.s[0] + dB[r][1] * R[j][1] * S.s[1] + dB[r][2] * R[j][2] * S.s[2];
        dRS[r][j] = C.Tcw[0 * 4 + r] * dB[0][j] + C.Tcw[1 * 4 + r] * dB[1][j] + C.Tcw[2 * 4 + r] * dB[2][j];
      }
    T d_ls[3], dR[3][3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      T dsj = R[0][j] * dRS[0][j] + R[1][j] * dRS[1][j] + R[2][j] * dRS[2][j];
      d_ls[j] = dsj * S.s[j];
#pragma unroll
      for (int r = 0; r < 3; ++r) dR[r][j] = dRS[r][j] * S.s[j];
    }
    // 6. R(q_hat), q_hat = q / |q|
    T dqx = dR[0][1] * T(2) * y + dR[0][2] * T(2) * z + dR[1][0] * T(2) * y - dR[1][1] * T(4) * x -
            dR[1][2] * T(2) * w + dR[2][0] * T(2) * z + dR[2][1] * T(2) * w - dR[2][2] * T(4) * x;
    T dqy = -dR[0][0] * T(4) * y + dR[0][1] * T(2) * x + dR[0][2] * T(2) * w + dR[1][0] * T(2) * x +
            dR[1][2] * T(2) * z - dR[2][0] * T(2) * w + dR[2][1] * T(2) * z - dR[2][2] * T(4) * y;
    T dqz = -dR[0][0] * T(4) * z - dR[0][1] * T(2) * w + dR[0][2] * T(2) * x + dR[1][0] * T(2) * w -
            dR[1][1] * T(4) * z + dR[1][2] * T(2) * y + dR[2][0] * T(2) * x + dR[2][1] * T(2) * y;
    T dqw = -dR[0][1] * T(2) * z + dR[0][2] * T(2) * y + dR[1][0] * T(2) * z - dR[1][2] * T(2) * x -
            dR[2][0] * T(2) * y + dR[2][1] * T(2) * x;
    T qd = x * dqx + y * dqy + z * dqz + w * dqw;
    T d_rot[4] = {(dqx - x * qd) / S.qn, (dqy - y * qd) / S.qn, (dqz - z * qd) / S.qn, (dqw - w * qd) / S.qn};
    // 7. jacobian entries
    const T iz = T(1) / zc, iz2 = iz * iz;
    T dfx = dJ00 * iz, dfy = dJ11 * iz;
    T dz = (-(dJ00 * C.fx + dJ11 * C.fy) + dJ02 * (S.tu - C.cx) + dJ12 * (S.tv - C.cy)) * iz2;
    T dtu = -dJ02 * iz, dtv = -dJ12 * iz;
    T dcx = dJ02 * iz, dcy = dJ12 * iz;
    // 8. clamp passes gradient strictly inside
    T du = d_mean_x + ((S.u > C.lo_x && S.u < C.hi_x) ? dtu : T(0));
    T dv = d_mean_y + ((S.v > C.lo_y && S.v < C.hi_y) ? dtv : T(0));
    // 9. u = fx x / z + cx
    const T xc = S.cam[0], yc = S.cam[1];
    dfx += du * xc * iz; dcx += du;
    dfy += dv * yc * iz; dcy += dv;
    T dxc = du * C.fx * iz, dyc = dv * C.fy * iz;
    dz += -(du * C.fx * xc + dv * C.fy * yc) * iz2 + d_depth;
    // 10. cam = W p + t
    T dcam[3] = {dxc, dyc, dz};
    T d_pos[3];
#pragma unroll
    for (int j = 0; j < 3; ++j)
      d_pos[j] = C.Tcw[0 * 4 + j] * dcam[0] + C.Tcw[1 * 4 + j] * dcam[1] + C.Tcw[2 * 4 + j] * dcam[2];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
#pragma unroll
      for (int j = 0; j < 3; ++j) cam_grad[r * 4 + j] += dcam[r] * pos[j];
      cam_grad[r * 4 + 3] += dcam[r];
    }
    cam_grad[12] = dfx; cam_grad[13] = dfy; cam_grad[14] = dcx; cam_grad[15] = dcy;

    // ACC: rows are unique, so a reduction without return value (red.global.add, resolved at the L2) gives the same
    // sum as a read-modify-write and the thread does not wait for eleven loads at its very end
    auto put = [](T* dst, T v) { if (ACC) red_add(dst, v); else *dst = v; };
    if (g_position) {
#pragma unroll
      for (int k = 0; k < 3; ++k) put(g_position + 3 * idx + k, d_pos[k]);
    }
    if (g_log_scaling) {
#pragma unroll
      for (int k = 0; k < 3; ++k) put(g_log_scaling + 3 * idx + k, d_ls[k]);
    }
    if (g_rotation) {
#pragma unroll
      for (int k = 0; k < 4; ++k) put(g_rotation + 4 * idx + k, d_rot[k]);
    }
    if (g_alpha_logit) put(g_alpha_logit + idx, d_logit);
  }

  if (g_Tcw || g_proj) {  // camera gradients are summed over gaussians (expand backward, projection.py:212-213)
    __shared__ T s_red[16][kPBwdBlock / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      T v = warp_sum(cam_grad[k]);
      if (lane == 0) s_red[k][warp] = v;
    }
    __syncthreads();
    if (threadIdx.x < 16) {
      T t = T(0);
#pragma unroll
      for (int wi = 0; wi < kPBwdBlock / 32; ++wi) t += s_red[threadIdx.x][wi];
      if (threadIdx.x < 12) { if (g_Tcw && t != T(0)) red_add(g_Tcw + threadIdx.x, t); }
      else if (g_proj && t != T(0)) red_add(g_proj + (threadIdx.x - 12), t);
    }
  }
}

}  // namespace gs

using namespace gs;

template <typename T>
static int sh_dispatch(bool backward, const GsSHParams* p, const void* params, const void* positions,
                       const int64_t* indexes, const void* cam, const void* grad_out, void* out_or_gparams,
                       void* gpos, void* gcam, cudaStream_t st, const int32_t* count_dev = nullptr) {
  const int64_t blocks = ceil_div(p->num_indexes, 256);
#define GS_SH_CASE(DD)                                                                                              \
  case DD:                                                                                                          \
    if (!backward)                                                                                                  \
      sh_fwd_kernel<T, DD><<<(unsigned)blocks, 256, 0, st>>>(*p, (const T*)params, (const T*)positions, indexes,    \
                                                             (const T*)cam, (T*)out_or_gparams, count_dev);         \
    else                                                                                                            \
      sh_bwd_kernel<T, DD><<<(unsigned)blocks, 256, 0, st>>>(*p, (const T*)params, (const T*)positions, indexes,    \
                                                             (const T*)cam, (const T*)grad_out, (T*)out_or_gparams, \
                                                             (T*)gpos, (T*)gcam);                                   \
    break;
  switch (p->num_coeffs) {
    GS_SH_CASE(1)
    GS_SH_CASE(4)
    GS_SH_CASE(9)
    GS_SH_CASE(16)
    default:
      GS_UNSUPPORTED("spherical harmonics: %d coefficients (degree must be 0..3)", p->num_coeffs);
  }
#undef GS_SH_CASE
  GS_LAUNCH_CHECK();
  return GS_OK;
}

static int check_sh(const GsSHParams* p, const char* who) {
  if (!p) { set_error("%s: null params", who); return GS_ERR_INVALID; }
  if (p->dtype != GS_F32 && p->dtype != GS_F64) { set_error("%s: bad dtype", who); return GS_ERR_INVALID; }
  if (p->num_channels <= 0 || p->num_points < 0 || p->num_indexes < 0) { set_error("%s: bad sizes", who); return GS_ERR_INVALID; }
  return GS_OK;
}

// The shapes the batched forward, the flush and the dense backward serve: f32, K = 3, degree 0..3
static bool sh_fast_shape(const GsSHParams* p) {
  return p->dtype == GS_F32 && p->num_channels == 3 &&
         (p->num_coeffs == 1 || p->num_coeffs == 4 || p->num_coeffs == 9 || p->num_coeffs == 16);
}

static bool aligned16(const void* ptr) { return ((uintptr_t)ptr & 15) == 0; }

template <int D, bool A16>
static void launch_sh_dense(bool fill, bool from_out, const GsSHParams* p, const void* params, const void* positions,
                            const int64_t* indexes, const void* cam, const void* grad_out, void* grad_params,
                            void* grad_positions, void* grad_cam, cudaStream_t st) {
  const unsigned blocks = (unsigned)ceil_div(p->num_indexes, kSHDenseBlock);
#define GS_SH_DENSE(FILLV, FROMV)                                                                                  \
  sh_bwd_dense_kernel<3, D, FILLV, FROMV, A16><<<blocks, kSHDenseBlock, 0, st>>>(                                 \
      *p, (const float*)params, (const float*)positions, indexes, (const float*)cam, (const float*)grad_out,       \
      (float*)grad_params, (float*)grad_positions, (float*)grad_cam)
  if (fill) { if (from_out) GS_SH_DENSE(true, true); else GS_SH_DENSE(true, false); }
  else { if (from_out) GS_SH_DENSE(false, true); else GS_SH_DENSE(false, false); }
#undef GS_SH_DENSE
}

template <int D, bool A16>
static void launch_sh_flush(bool overwrite, int64_t n, int num_views, const SHFlushViews& views, const void* positions,
                            void* grad_params, cudaStream_t st) {
  const unsigned blocks = (unsigned)ceil_div(n, kSHDenseBlock);
  if (overwrite)
    sh_bwd_flush_kernel<3, D, true, A16><<<blocks, kSHDenseBlock, 0, st>>>(n, num_views, views, (const float*)positions,
                                                                            (float*)grad_params);
  else
    sh_bwd_flush_kernel<3, D, false, A16><<<blocks, kSHDenseBlock, 0, st>>>(n, num_views, views, (const float*)positions,
                                                                             (float*)grad_params);
}

template <int D, bool A16>
static void launch_sh_fwd_views(int64_t n, int num_views, const SHViewsOut& views, const void* params,
                                const void* positions, cudaStream_t st) {
  sh_fwd_views_kernel<3, D, A16><<<(unsigned)ceil_div(n, 128), 128, 0, st>>>(n, num_views, views, (const float*)params,
                                                                             (const float*)positions);
}

extern "C" {

int gs_sh_fwd(const GsSHParams* p, const void* params, const void* positions, const int64_t* indexes,
              const void* camera_pos, void* out, void* stream) {
  int rc = check_sh(p, "gs_sh_fwd");
  if (rc != GS_OK) return rc;
  if (p->num_indexes == 0) return GS_OK;
  GS_CHECK_ARG(params && positions && indexes && camera_pos && out, "gs_sh_fwd: null tensor");
  cudaStream_t st = (cudaStream_t)stream;
  return p->dtype == GS_F32
             ? sh_dispatch<float>(false, p, params, positions, indexes, camera_pos, nullptr, out, nullptr, nullptr, st)
             : sh_dispatch<double>(false, p, params, positions, indexes, camera_pos, nullptr, out, nullptr, nullptr, st);
}

int gs_sh_fwd_counted(const GsSHParams* p, const void* params, const void* positions, const int64_t* indexes,
                      const void* camera_pos, const int32_t* count_dev, void* out, void* stream) {
  int rc = check_sh(p, "gs_sh_fwd_counted");
  if (rc != GS_OK) return rc;
  if (p->num_indexes == 0) return GS_OK;
  GS_CHECK_ARG(params && positions && indexes && camera_pos && out && count_dev, "gs_sh_fwd_counted: null tensor");
  cudaStream_t st = (cudaStream_t)stream;
  return p->dtype == GS_F32 ? sh_dispatch<float>(false, p, params, positions, indexes, camera_pos, nullptr, out, nullptr,
                                                 nullptr, st, count_dev)
                            : sh_dispatch<double>(false, p, params, positions, indexes, camera_pos, nullptr, out,
                                                  nullptr, nullptr, st, count_dev);
}

int gs_sh_bwd(const GsSHParams* p, const void* params, const void* positions, const int64_t* indexes,
              const void* camera_pos, const void* grad_out, void* grad_params, void* grad_positions,
              void* grad_camera_pos, void* stream) {
  int rc = check_sh(p, "gs_sh_bwd");
  if (rc != GS_OK) return rc;
  if (p->accumulate_params != 0) {
    set_error("gs_sh_bwd: accumulate_params is reserved and must be 0, got %d", p->accumulate_params);
    return GS_ERR_INVALID;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const size_t es = p->dtype == GS_F32 ? 4 : 8;
  const bool dense = p->indexes_sorted_unique && grad_params != nullptr && p->num_indexes > 0 && sh_fast_shape(p);
  const bool from_out = p->params_is_forward_output != 0;
  if (from_out && (!dense || grad_positions || grad_camera_pos)) {
    set_error("gs_sh_bwd: params_is_forward_output needs the dense path and no position / camera gradient");
    return GS_ERR_UNSUPPORTED;
  }
  const bool fill = dense && 2 * p->num_indexes >= p->num_points;  // mostly visible: zero-fill the gaps in-kernel
  if (grad_params && !fill)
    GS_CUDA(cudaMemsetAsync(grad_params, 0, (size_t)p->num_points * p->num_channels * p->num_coeffs * es, st));
  if (grad_positions && !fill) GS_CUDA(cudaMemsetAsync(grad_positions, 0, (size_t)p->num_points * 3 * es, st));
  if (grad_camera_pos) GS_CUDA(cudaMemsetAsync(grad_camera_pos, 0, 3 * es, st));
  if (p->num_indexes == 0) return GS_OK;
  GS_CHECK_ARG(params && positions && indexes && camera_pos && grad_out, "gs_sh_bwd: null tensor");
  if (dense) {
    // 16 B units where the rows allow them (D = 4, 16) and the pointers they go through are 16 B aligned
    const bool a16 = aligned16(grad_params) && (from_out || aligned16(params));
#define GS_SH_DENSE_ARGS fill, from_out, p, params, positions, indexes, camera_pos, grad_out, grad_params, \
                         grad_positions, grad_camera_pos, st
    switch (p->num_coeffs) {
      case 1: launch_sh_dense<1, false>(GS_SH_DENSE_ARGS); break;
      case 4: if (a16) launch_sh_dense<4, true>(GS_SH_DENSE_ARGS); else launch_sh_dense<4, false>(GS_SH_DENSE_ARGS); break;
      case 9: launch_sh_dense<9, false>(GS_SH_DENSE_ARGS); break;
      default: if (a16) launch_sh_dense<16, true>(GS_SH_DENSE_ARGS); else launch_sh_dense<16, false>(GS_SH_DENSE_ARGS);
    }
#undef GS_SH_DENSE_ARGS
    GS_LAUNCH_CHECK();
    return GS_OK;
  }
  return p->dtype == GS_F32 ? sh_dispatch<float>(true, p, params, positions, indexes, camera_pos, grad_out,
                                                 grad_params, grad_positions, grad_camera_pos, st)
                            : sh_dispatch<double>(true, p, params, positions, indexes, camera_pos, grad_out,
                                                  grad_params, grad_positions, grad_camera_pos, st);
}

static int sh_bwd_stage_entry(const GsSHParams* p, const void* forward_out, const int64_t* indexes, const void* grad_out,
                             const int32_t* count_dev, void* staged, void* stream) {
  int rc = check_sh(p, "gs_sh_bwd_stage");
  if (rc != GS_OK) return rc;
  if (p->dtype != GS_F32 || p->num_channels != 3) {
    set_error("gs_sh_bwd_stage: f32 and K = 3 only");
    return GS_ERR_UNSUPPORTED;
  }
  GS_CHECK_ARG(staged != nullptr, "gs_sh_bwd_stage: null staging buffer");
  cudaStream_t st = (cudaStream_t)stream;
  if (count_dev != nullptr || p->num_indexes < p->num_points)   // culled gaussians stage zeros
    GS_CUDA(cudaMemsetAsync(staged, 0, (size_t)p->num_points * 3 * sizeof(float), st));
  if (p->num_indexes == 0) return GS_OK;
  GS_CHECK_ARG(forward_out && indexes && grad_out, "gs_sh_bwd_stage: null tensor");
  sh_bwd_stage_kernel<3><<<(unsigned)ceil_div(p->num_indexes, 256), 256, 0, st>>>(
      p->num_indexes, (const float*)forward_out, indexes, (const float*)grad_out, (float*)staged, count_dev);
  GS_LAUNCH_CHECK();
  return GS_OK;
}

int gs_sh_bwd_stage(const GsSHParams* p, const void* forward_out, const int64_t* indexes, const void* grad_out,
                    void* staged, void* stream) {
  return sh_bwd_stage_entry(p, forward_out, indexes, grad_out, nullptr, staged, stream);
}

int gs_sh_bwd_stage_counted(const GsSHParams* p, const void* forward_out, const int64_t* indexes, const void* grad_out,
                            const int32_t* count_dev, void* staged, void* stream) {
  GS_CHECK_ARG(count_dev != nullptr, "gs_sh_bwd_stage_counted: null count");
  return sh_bwd_stage_entry(p, forward_out, indexes, grad_out, count_dev, staged, stream);
}

int gs_sh_bwd_flush(const GsSHParams* p, int32_t num_views, const void* const* staged,
                    const void* const* camera_positions, const void* positions, void* grad_params, void* stream) {
  GS_CHECK_ARG(p != nullptr, "gs_sh_bwd_flush: null params");
  if (!sh_fast_shape(p)) {
    set_error("gs_sh_bwd_flush: f32, K = 3 and D in {1, 4, 9, 16} only (got dtype %d, K = %d, D = %d)", p->dtype,
              p->num_channels, p->num_coeffs);
    return GS_ERR_UNSUPPORTED;
  }
  GS_CHECK_ARG(num_views >= 0 && num_views <= kSHMaxDeferred, "gs_sh_bwd_flush: at most 16 views per flush");
  const bool overwrite = p->accumulate_params == 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (p->num_points == 0) return GS_OK;
  if (num_views == 0) {
    if (overwrite) {
      GS_CHECK_ARG(grad_params != nullptr, "gs_sh_bwd_flush: null tensor");
      GS_CUDA(cudaMemsetAsync(grad_params, 0, (size_t)p->num_points * 3 * p->num_coeffs * sizeof(float), st));
    }
    return GS_OK;
  }
  GS_CHECK_ARG(staged && camera_positions && positions && grad_params, "gs_sh_bwd_flush: null tensor");
  SHFlushViews views;
  for (int v = 0; v < kSHMaxDeferred; ++v) {
    views.staged[v] = v < num_views ? (const float*)staged[v] : nullptr;
    views.cam[v] = v < num_views ? (const float*)camera_positions[v] : nullptr;
    GS_CHECK_ARG(v >= num_views || (views.staged[v] && views.cam[v]), "gs_sh_bwd_flush: null view");
  }
  // float4 units when grad_params is 16 B aligned (a bucket slice after an odd parameter count is only 4 B aligned)
  const bool a16 = aligned16(grad_params);
#define GS_SH_FLUSH_ARGS overwrite, p->num_points, num_views, views, positions, grad_params, st
  switch (p->num_coeffs) {
    case 1: if (a16) launch_sh_flush<1, true>(GS_SH_FLUSH_ARGS); else launch_sh_flush<1, false>(GS_SH_FLUSH_ARGS); break;
    case 4: if (a16) launch_sh_flush<4, true>(GS_SH_FLUSH_ARGS); else launch_sh_flush<4, false>(GS_SH_FLUSH_ARGS); break;
    case 9: if (a16) launch_sh_flush<9, true>(GS_SH_FLUSH_ARGS); else launch_sh_flush<9, false>(GS_SH_FLUSH_ARGS); break;
    default: if (a16) launch_sh_flush<16, true>(GS_SH_FLUSH_ARGS); else launch_sh_flush<16, false>(GS_SH_FLUSH_ARGS);
  }
#undef GS_SH_FLUSH_ARGS
  GS_LAUNCH_CHECK();
  return GS_OK;
}

int gs_sh_fwd_views(const GsSHParams* p, int32_t num_views, const void* params, const void* positions,
                    const void* const* camera_positions, void* const* outs, void* stream) {
  GS_CHECK_ARG(p != nullptr, "gs_sh_fwd_views: null params");
  if (!sh_fast_shape(p)) {
    set_error("gs_sh_fwd_views: f32, K = 3 and D in {1, 4, 9, 16} only (got dtype %d, K = %d, D = %d)", p->dtype,
              p->num_channels, p->num_coeffs);
    return GS_ERR_UNSUPPORTED;
  }
  GS_CHECK_ARG(num_views >= 0 && num_views <= kSHMaxDeferred, "gs_sh_fwd_views: at most 16 views per call");
  if (num_views == 0 || p->num_points == 0) return GS_OK;
  GS_CHECK_ARG(params && positions && camera_positions && outs, "gs_sh_fwd_views: null tensor");
  SHViewsOut views;
  for (int v = 0; v < kSHMaxDeferred; ++v) {
    views.out[v] = v < num_views ? (float*)outs[v] : nullptr;
    views.cam[v] = v < num_views ? (const float*)camera_positions[v] : nullptr;
    GS_CHECK_ARG(v >= num_views || (views.out[v] && views.cam[v]), "gs_sh_fwd_views: null view");
  }
  cudaStream_t st = (cudaStream_t)stream;
  const bool a16 = aligned16(params);   // float4 rows at D = 4, 16; rows of 3 or 27 floats are read one float at a time
#define GS_SH_VIEWS_ARGS p->num_points, num_views, views, params, positions, st
  switch (p->num_coeffs) {
    case 1: launch_sh_fwd_views<1, false>(GS_SH_VIEWS_ARGS); break;
    case 4: if (a16) launch_sh_fwd_views<4, true>(GS_SH_VIEWS_ARGS); else launch_sh_fwd_views<4, false>(GS_SH_VIEWS_ARGS); break;
    case 9: launch_sh_fwd_views<9, false>(GS_SH_VIEWS_ARGS); break;
    default:
      if (a16) launch_sh_fwd_views<16, true>(GS_SH_VIEWS_ARGS); else launch_sh_fwd_views<16, false>(GS_SH_VIEWS_ARGS);
  }
#undef GS_SH_VIEWS_ARGS
  GS_LAUNCH_CHECK();
  return GS_OK;
}

int gs_gather_rows_counted(int64_t capacity, int32_t row_floats, const void* src, const int64_t* indexes,
                           const int32_t* count_dev, void* out, void* stream) {
  GS_CHECK_ARG(capacity >= 0, "gs_gather_rows_counted: bad capacity");
  if (row_floats != 3) {
    set_error("gs_gather_rows_counted: rows of 3 floats only");
    return GS_ERR_UNSUPPORTED;
  }
  if (capacity == 0) return GS_OK;
  GS_CHECK_ARG(src && indexes && out, "gs_gather_rows_counted: null tensor");
  gather_rows_counted_kernel<3><<<(unsigned)ceil_div(capacity, 256), 256, 0, (cudaStream_t)stream>>>(
      capacity, (const float*)src, indexes, count_dev, (float*)out);
  GS_LAUNCH_CHECK();
  return GS_OK;
}

}  // extern "C"

template <typename T>
static int gather_rows_strided(const char* who, int64_t capacity, int32_t row_floats, const T* src,
                               const int64_t* indexes, const int32_t* count_dev, T* out, int32_t out_stride,
                               int32_t out_offset, void* stream) {
  GS_CHECK_ARG(capacity >= 0 && row_floats > 0 && out_offset >= 0 && out_stride >= out_offset + row_floats,
               "%s: bad sizes", who);
  if (capacity == 0) return GS_OK;
  GS_CHECK_ARG(src && indexes && out, "%s: null tensor", who);
  const int64_t total = capacity * row_floats;
  if (total + 256 < (1ll << 32))
    gather_rows_strided_kernel<uint32_t, T><<<(unsigned)ceil_div(total, 256), 256, 0, (cudaStream_t)stream>>>(
        capacity, row_floats, src, indexes, count_dev, out, out_stride, out_offset);
  else
    gather_rows_strided_kernel<uint64_t, T><<<(unsigned)ceil_div(total, 256), 256, 0, (cudaStream_t)stream>>>(
        capacity, row_floats, src, indexes, count_dev, out, out_stride, out_offset);
  GS_LAUNCH_CHECK();
  return GS_OK;
}

template <typename T>
static int scatter_rows_strided(const char* who, int64_t capacity, int32_t row_floats, const T* src, int32_t src_stride,
                                int32_t src_offset, const int64_t* indexes, const int32_t* count_dev, int64_t dst_rows,
                                T* dst, void* stream) {
  GS_CHECK_ARG(capacity >= 0 && row_floats > 0 && src_offset >= 0 && src_stride >= src_offset + row_floats &&
                   dst_rows >= 0, "%s: bad sizes", who);
  if (dst_rows == 0) return GS_OK;
  GS_CHECK_ARG(dst != nullptr, "%s: null destination", who);
  cudaStream_t st = (cudaStream_t)stream;
  GS_CUDA(cudaMemsetAsync(dst, 0, (size_t)dst_rows * row_floats * sizeof(T), st));   // rows outside the visible set
  if (capacity == 0) return GS_OK;
  GS_CHECK_ARG(src && indexes, "%s: null tensor", who);
  const int64_t total = capacity * row_floats;
  if (total + 256 < (1ll << 32))
    scatter_rows_strided_kernel<uint32_t, T><<<(unsigned)ceil_div(total, 256), 256, 0, st>>>(
        capacity, row_floats, src, src_stride, src_offset, indexes, count_dev, dst);
  else
    scatter_rows_strided_kernel<uint64_t, T><<<(unsigned)ceil_div(total, 256), 256, 0, st>>>(
        capacity, row_floats, src, src_stride, src_offset, indexes, count_dev, dst);
  GS_LAUNCH_CHECK();
  return GS_OK;
}

extern "C" {

int gs_gather_rows_strided(int64_t capacity, int32_t row_floats, const float* src, const int64_t* indexes,
                           const int32_t* count_dev, float* out, int32_t out_stride, int32_t out_offset, void* stream) {
  return gather_rows_strided("gs_gather_rows_strided", capacity, row_floats, src, indexes, count_dev, out, out_stride,
                             out_offset, stream);
}

int gs_scatter_rows_strided(int64_t capacity, int32_t row_floats, const float* src, int32_t src_stride,
                            int32_t src_offset, const int64_t* indexes, const int32_t* count_dev, int64_t dst_rows,
                            float* dst, void* stream) {
  return scatter_rows_strided("gs_scatter_rows_strided", capacity, row_floats, src, src_stride, src_offset, indexes,
                              count_dev, dst_rows, dst, stream);
}

int gs_gather_rows_strided_u16(int64_t capacity, int32_t row_elems, const uint16_t* src, const int64_t* indexes,
                               const int32_t* count_dev, uint16_t* out, int32_t out_stride, int32_t out_offset,
                               void* stream) {
  return gather_rows_strided("gs_gather_rows_strided_u16", capacity, row_elems, src, indexes, count_dev, out,
                             out_stride, out_offset, stream);
}

int gs_scatter_rows_strided_u16(int64_t capacity, int32_t row_elems, const uint16_t* src, int32_t src_stride,
                                int32_t src_offset, const int64_t* indexes, const int32_t* count_dev, int64_t dst_rows,
                                uint16_t* dst, void* stream) {
  return scatter_rows_strided("gs_scatter_rows_strided_u16", capacity, row_elems, src, src_stride, src_offset,
                              indexes, count_dev, dst_rows, dst, stream);
}

int gs_split_channels(int64_t rows, int32_t channels, int32_t split, const float* src, float* first, float* rest,
                      void* stream) {
  GS_CHECK_ARG(rows >= 0 && channels > 0 && split > 0 && split < channels, "gs_split_channels: bad sizes");
  if (rows == 0) return GS_OK;
  GS_CHECK_ARG(src && first && rest, "gs_split_channels: null tensor");
  const int64_t total = rows * channels;
  const bool small = total + 512 < (1ll << 32);
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned g2 = (unsigned)ceil_div(total / 2, 256), g1 = (unsigned)ceil_div(total, 256);
  if (channels % 2 == 0 && split % 2 == 0) {
    if (small) split_channels_kernel<2, uint32_t><<<g2, 256, 0, st>>>(total, channels, split, src, first, rest);
    else split_channels_kernel<2, uint64_t><<<g2, 256, 0, st>>>(total, channels, split, src, first, rest);
  } else {
    if (small) split_channels_kernel<1, uint32_t><<<g1, 256, 0, st>>>(total, channels, split, src, first, rest);
    else split_channels_kernel<1, uint64_t><<<g1, 256, 0, st>>>(total, channels, split, src, first, rest);
  }
  GS_LAUNCH_CHECK();
  return GS_OK;
}

int gs_merge_channels(int64_t rows, int32_t channels, int32_t split, const float* first, const float* rest, float* dst,
                      void* stream) {
  GS_CHECK_ARG(rows >= 0 && channels > 0 && split > 0 && split < channels, "gs_merge_channels: bad sizes");
  if (rows == 0) return GS_OK;
  GS_CHECK_ARG(dst != nullptr, "gs_merge_channels: null destination");
  const int64_t total = rows * channels;
  const bool small = total + 512 < (1ll << 32);
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned g2 = (unsigned)ceil_div(total / 2, 256), g1 = (unsigned)ceil_div(total, 256);
  if (channels % 2 == 0 && split % 2 == 0) {
    if (small) merge_channels_kernel<2, uint32_t><<<g2, 256, 0, st>>>(total, channels, split, first, rest, dst);
    else merge_channels_kernel<2, uint64_t><<<g2, 256, 0, st>>>(total, channels, split, first, rest, dst);
  } else {
    if (small) merge_channels_kernel<1, uint32_t><<<g1, 256, 0, st>>>(total, channels, split, first, rest, dst);
    else merge_channels_kernel<1, uint64_t><<<g1, 256, 0, st>>>(total, channels, split, first, rest, dst);
  }
  GS_LAUNCH_CHECK();
  return GS_OK;
}

static int project_bwd_entry(const GsProjectParams* p, int64_t num_visible, const int32_t* count_dev,
                             const void* position, const void* log_scaling,
                   const void* rotation, const void* alpha_logit, const void* T_camera_world, const void* projection,
                   const int64_t* indexes, const void* grad_points, const void* grad_depth, void* grad_position,
                   void* grad_log_scaling, void* grad_rotation, void* grad_alpha_logit, void* grad_T_camera_world,
                   void* grad_projection, void* stream) {
  GS_CHECK_ARG(p != nullptr, "gs_project_bwd: null params");
  GS_CHECK_ARG(p->dtype == GS_F32 || p->dtype == GS_F64, "gs_project_bwd: bad dtype");
  GS_CHECK_ARG(num_visible >= 0 && num_visible <= p->num_points, "gs_project_bwd: bad num_visible");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t es = p->dtype == GS_F32 ? 4 : 8;
  const size_t n = (size_t)p->num_points;
  const bool acc = p->accumulate_grads != 0;
  if (!acc) {
    if (grad_position) GS_CUDA(cudaMemsetAsync(grad_position, 0, n * 3 * es, st));
    if (grad_log_scaling) GS_CUDA(cudaMemsetAsync(grad_log_scaling, 0, n * 3 * es, st));
    if (grad_rotation) GS_CUDA(cudaMemsetAsync(grad_rotation, 0, n * 4 * es, st));
    if (grad_alpha_logit) GS_CUDA(cudaMemsetAsync(grad_alpha_logit, 0, n * es, st));
  }
  if (grad_T_camera_world) GS_CUDA(cudaMemsetAsync(grad_T_camera_world, 0, 16 * es, st));
  if (grad_projection) GS_CUDA(cudaMemsetAsync(grad_projection, 0, 4 * es, st));
  if (num_visible == 0) return GS_OK;
  GS_CHECK_ARG(position && log_scaling && rotation && alpha_logit && T_camera_world && projection && indexes &&
                   grad_points, "gs_project_bwd: null tensor");
  const int64_t blocks = ceil_div(num_visible, kPBwdBlock);
#define GS_PBWD_LAUNCH(TT, ACCV)                                                                                    \
  project_bwd_kernel<TT, ACCV><<<(unsigned)blocks, kPBwdBlock, 0, st>>>(                                            \
      *p, num_visible, (const TT*)position, (const TT*)log_scaling, (const TT*)rotation, (const TT*)alpha_logit,    \
      (const TT*)T_camera_world, (const TT*)projection, indexes, (const TT*)grad_points, (const TT*)grad_depth,     \
      (TT*)grad_position, (TT*)grad_log_scaling, (TT*)grad_rotation, (TT*)grad_alpha_logit,                         \
      (TT*)grad_T_camera_world, (TT*)grad_projection, count_dev)
  if (p->dtype == GS_F32) { if (acc) GS_PBWD_LAUNCH(float, true); else GS_PBWD_LAUNCH(float, false); }
  else { if (acc) GS_PBWD_LAUNCH(double, true); else GS_PBWD_LAUNCH(double, false); }
#undef GS_PBWD_LAUNCH
  GS_LAUNCH_CHECK();
  return GS_OK;
}

int gs_project_bwd(const GsProjectParams* p, int64_t num_visible, const void* position, const void* log_scaling,
                   const void* rotation, const void* alpha_logit, const void* T_camera_world, const void* projection,
                   const int64_t* indexes, const void* grad_points, const void* grad_depth, void* grad_position,
                   void* grad_log_scaling, void* grad_rotation, void* grad_alpha_logit, void* grad_T_camera_world,
                   void* grad_projection, void* stream) {
  return project_bwd_entry(p, num_visible, nullptr, position, log_scaling, rotation, alpha_logit, T_camera_world,
                           projection, indexes, grad_points, grad_depth, grad_position, grad_log_scaling, grad_rotation,
                           grad_alpha_logit, grad_T_camera_world, grad_projection, stream);
}

int gs_project_bwd_counted(const GsProjectParams* p, int64_t capacity, const int32_t* count_dev, const void* position,
                           const void* log_scaling, const void* rotation, const void* alpha_logit,
                           const void* T_camera_world, const void* projection, const int64_t* indexes,
                           const void* grad_points, const void* grad_depth, void* grad_position,
                           void* grad_log_scaling, void* grad_rotation, void* grad_alpha_logit,
                           void* grad_T_camera_world, void* grad_projection, void* stream) {
  GS_CHECK_ARG(count_dev != nullptr, "gs_project_bwd_counted: null count");
  return project_bwd_entry(p, capacity, count_dev, position, log_scaling, rotation, alpha_logit, T_camera_world,
                           projection, indexes, grad_points, grad_depth, grad_position, grad_log_scaling, grad_rotation,
                           grad_alpha_logit, grad_T_camera_world, grad_projection, stream);
}

}  // extern "C"
