// Small-K softmax glue around the OCR (object-contextual representation) GEMMs.
//
// The two skinny products of SpatialGather (network/ocr_utils.py:34-46) and ObjectAttentionBlock
// (network/ocr_utils.py:95-119) run on the tcgen05 convolution / weight-gradient kernels with the 19 classes padded to
// a 32-wide bf16 operand; what remains here are the softmaxes between them (K = num_classes <= 32):
//   spatial softmax  : over the H*W pixels of each (image, class) map  -> probs bf16 [pixels][32]
//   class softmax    : over the classes of each pixel, with the key_channels^-0.5 scale -> sim bf16 [pixels][32]
// plus their backward passes and two layout helpers (transpose+pad, fp32->bf16 cast).
#include "ptx.cuh"
#include "launch.h"
#include "../../include/b200seg.h"
#include "vec.cuh"

namespace b200seg {

constexpr int KP = 32;   // padded class count of every bf16 class-operand

// ---------------------------------------------------------------------------------------- spatial softmax (over pixels)
// partial[n][b][k] = (max, sum exp(x - max)) over the block's pixel range
__global__ void __launch_bounds__(256)
spatial_stats_kernel(const float* __restrict__ x, int ld, int P, int K, float* __restrict__ partial) {
  pdl_sync();
  const int n = blockIdx.y, b = blockIdx.x, B = gridDim.x;
  const float* xn = x + (size_t)n * P * ld;
  float mx[KP], sm[KP];
#pragma unroll
  for (int k = 0; k < KP; ++k) { mx[k] = -INFINITY; sm[k] = 0.f; }
  for (int pix = b * 256 + threadIdx.x; pix < P; pix += B * 256) {
    const float* r = xn + (size_t)pix * ld;
#pragma unroll
    for (int k = 0; k < KP; ++k) {
      if (k < K) {
        const float v = r[k];
        if (v > mx[k]) { sm[k] = sm[k] * __expf(mx[k] - v) + 1.f; mx[k] = v; }
        else sm[k] += __expf(v - mx[k]);
      }
    }
  }
  __shared__ float s_m[8][KP], s_s[8][KP];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < KP; ++k) {
    float m = mx[k], s = sm[k];
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
      const float m2 = __shfl_xor_sync(0xffffffffu, m, off), s2 = __shfl_xor_sync(0xffffffffu, s, off);
      const float mm = fmaxf(m, m2);
      s = (m == -INFINITY ? 0.f : s * __expf(m - mm)) + (m2 == -INFINITY ? 0.f : s2 * __expf(m2 - mm));
      m = mm;
    }
    if (lane == 0) { s_m[warp][k] = m; s_s[warp][k] = s; }
  }
  __syncthreads();
  if (threadIdx.x < K) {
    const int k = threadIdx.x;
    float m = -INFINITY, s = 0.f;
    for (int w = 0; w < 8; ++w) {
      const float m2 = s_m[w][k], s2 = s_s[w][k];
      const float mm = fmaxf(m, m2);
      s = (m == -INFINITY ? 0.f : s * __expf(m - mm)) + (m2 == -INFINITY ? 0.f : s2 * __expf(m2 - mm));
      m = mm;
    }
    partial[(((size_t)n * B + b) * KP + k) * 2] = m;
    partial[(((size_t)n * B + b) * KP + k) * 2 + 1] = s;
  }
}

// probs[n][pix][k] = exp(x - max_k) / sum_k  (bf16, zero for k >= K); each block first folds the B partials.
__global__ void __launch_bounds__(256)
spatial_apply_kernel(const float* __restrict__ x, int ld, int P, int K, const float* __restrict__ partial, int B,
                     __nv_bfloat16* __restrict__ probs, float* __restrict__ stat_out) {
  pdl_sync();
  const int n = blockIdx.y;
  __shared__ float s_max[KP], s_inv[KP];
  if (threadIdx.x < KP) {
    const int k = threadIdx.x;
    float m = -INFINITY, s = 0.f;
    if (k < K) {
      for (int b = 0; b < B; ++b) {
        const float m2 = partial[(((size_t)n * B + b) * KP + k) * 2], s2 = partial[(((size_t)n * B + b) * KP + k) * 2 + 1];
        const float mm = fmaxf(m, m2);
        s = (m == -INFINITY ? 0.f : s * __expf(m - mm)) + (m2 == -INFINITY ? 0.f : s2 * __expf(m2 - mm));
        m = mm;
      }
    }
    s_max[k] = m;
    s_inv[k] = k < K ? 1.f / s : 0.f;
    if (stat_out && blockIdx.x == 0 && k < K) { stat_out[((size_t)n * KP + k) * 2] = m; stat_out[((size_t)n * KP + k) * 2 + 1] = s; }
  }
  __syncthreads();
  const float* xn = x + (size_t)n * P * ld;
  __nv_bfloat16* pn = probs + (size_t)n * P * KP;
  for (int pix = blockIdx.x * 256 + threadIdx.x; pix < P; pix += gridDim.x * 256) {
    const float* r = xn + (size_t)pix * ld;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int k = g * 8 + j;
        v[j] = k < K ? __expf(r[k] - s_max[k]) * s_inv[k] : 0.f;
      }
      store8(pn + (size_t)pix * KP + g * 8, v);
    }
  }
}

// backward: S[n][k] = sum_pix probs * dprobs  (block partials), then dlogit = probs * (dprobs - S)
__global__ void __launch_bounds__(256)
spatial_bwd_reduce_kernel(const float* __restrict__ dprobs, int ldd, const __nv_bfloat16* __restrict__ probs, int P,
                          int K, float* __restrict__ partial) {
  pdl_sync();
  const int n = blockIdx.y, b = blockIdx.x, B = gridDim.x;
  float acc[KP];
#pragma unroll
  for (int k = 0; k < KP; ++k) acc[k] = 0.f;
  for (int pix = b * 256 + threadIdx.x; pix < P; pix += B * 256) {
    const float* d = dprobs + ((size_t)n * P + pix) * ldd;
    const __nv_bfloat16* pr = probs + ((size_t)n * P + pix) * KP;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      float v[8];
      load8(pr + g * 8, v);
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (g * 8 + j < K) acc[g * 8 + j] += v[j] * d[g * 8 + j];
    }
  }
  __shared__ float s_a[8][KP];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < KP; ++k) {
    float a = acc[k];
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) a += __shfl_xor_sync(0xffffffffu, a, off);
    if (lane == 0) s_a[warp][k] = a;
  }
  __syncthreads();
  if (threadIdx.x < KP) {
    float a = 0.f;
    for (int w = 0; w < 8; ++w) a += s_a[w][threadIdx.x];
    partial[((size_t)n * B + b) * KP + threadIdx.x] = a;
  }
}

__global__ void __launch_bounds__(256)
spatial_bwd_apply_kernel(const float* __restrict__ dprobs, int ldd, const __nv_bfloat16* __restrict__ probs, int P, int K,
                         const float* __restrict__ partial, int B, __nv_bfloat16* __restrict__ dlogit, int accumulate) {
  pdl_sync();
  const int n = blockIdx.y;
  __shared__ float s_S[KP];
  if (threadIdx.x < KP) {
    float a = 0.f;
    for (int b = 0; b < B; ++b) a += partial[((size_t)n * B + b) * KP + threadIdx.x];
    s_S[threadIdx.x] = a;
  }
  __syncthreads();
  for (int pix = blockIdx.x * 256 + threadIdx.x; pix < P; pix += gridDim.x * 256) {
    const float* d = dprobs + ((size_t)n * P + pix) * ldd;
    const __nv_bfloat16* pr = probs + ((size_t)n * P + pix) * KP;
    __nv_bfloat16* o = dlogit + ((size_t)n * P + pix) * KP;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      float v[8], r[8];
      load8(pr + g * 8, v);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int k = g * 8 + j;
        r[j] = k < K ? v[j] * (d[k] - s_S[k]) : 0.f;
      }
      if (accumulate) {
        float old[8];
        load8(o + g * 8, old);
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] += old[j];
      }
      store8(o + g * 8, r);
    }
  }
}

// ---------------------------------------------------------------------------------------- class softmax (per pixel)
__global__ void __launch_bounds__(256)
class_softmax_fwd_kernel(const float* __restrict__ x, int ld, long long P, int K, float scale,
                         __nv_bfloat16* __restrict__ sim) {
  pdl_sync();
  for (long long pix = (long long)blockIdx.x * 256 + threadIdx.x; pix < P; pix += (long long)gridDim.x * 256) {
    const float* r = x + pix * ld;
    float v[KP];
    float m = -INFINITY;
#pragma unroll
    for (int k = 0; k < KP; ++k) {
      v[k] = k < K ? r[k] * scale : -INFINITY;
      m = fmaxf(m, v[k]);
    }
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < KP; ++k) { v[k] = k < K ? __expf(v[k] - m) : 0.f; s += v[k]; }
    const float inv = 1.f / s;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = v[g * 8 + j] * inv;
      store8(sim + pix * KP + g * 8, o);
    }
  }
}

// ds = scale * sim * (dsim - sum_k sim*dsim)
__global__ void __launch_bounds__(256)
class_softmax_bwd_kernel(const float* __restrict__ dsim, int ld, const __nv_bfloat16* __restrict__ sim, long long P,
                         int K, float scale, __nv_bfloat16* __restrict__ ds) {
  pdl_sync();
  for (long long pix = (long long)blockIdx.x * 256 + threadIdx.x; pix < P; pix += (long long)gridDim.x * 256) {
    const float* d = dsim + pix * ld;
    float s[KP], g[KP];
    float dot = 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float v[8];
      load8(sim + pix * KP + q * 8, v);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int k = q * 8 + j;
        s[k] = v[j];
        g[k] = k < K ? d[k] : 0.f;
        dot += s[k] * g[k];
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int k = q * 8 + j;
        o[j] = k < K ? scale * s[k] * (g[k] - dot) : 0.f;
      }
      store8(ds + pix * KP + q * 8, o);
    }
  }
}

// ---------------------------------------------------------------------------------------- layout helpers
// dst[c][r] (pitch rpad, zero padded) = src[r][c]   (src bf16 [R][C] with pitch ld, or fp32 when src_fp32)
__global__ void transpose_pad_kernel(const void* __restrict__ src, int src_fp32, int R, int C, int ld,
                                     __nv_bfloat16* __restrict__ dst, int rpad) {
  pdl_sync();
  const int total = C * rpad;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int c = i / rpad, r = i - c * rpad;
    float v = 0.f;
    if (r < R)
      v = src_fp32 ? reinterpret_cast<const float*>(src)[(size_t)r * ld + c]
                   : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(src)[(size_t)r * ld + c]);
    dst[i] = __float2bfloat16_rn(v);
  }
}

// dst bf16 [rows][dst_ld] = (accumulate? dst : 0) + src fp32 [rows][src_ld] for cols < C
__global__ void cast_rows_kernel(const float* __restrict__ src, int src_ld, __nv_bfloat16* __restrict__ dst, int dst_ld,
                                 long long rows, int C, int accumulate) {
  pdl_sync();
  const long long total = rows * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / C;
    const int c = (int)(i - r * C);
    float v = src[r * src_ld + c];
    if (accumulate) v += __bfloat162float(dst[r * dst_ld + c]);
    dst[r * dst_ld + c] = __float2bfloat16_rn(v);
  }
}


// partials[block][c] = sum over the block's rows of dy[row][c] for c < C (conv bias gradient of the logit heads; dy bf16
// [rows][ld]). The blocks' sums are combined by colsum_finish_kernel in a fixed order, not with atomics, so the gradient
// is the same bit for bit on every run.
__global__ void __launch_bounds__(256)
colsum_kernel(const __nv_bfloat16* __restrict__ dy, int ld, long long rows, int C, float* __restrict__ partials) {
  pdl_sync();
  // thread (r, c): 8 row-lanes x 32 columns
  const int c = threadIdx.x & 31, r = threadIdx.x >> 5;
  float acc = 0.f;
  if (c < C)
    for (long long row = (long long)blockIdx.x * 8 + r; row < rows; row += (long long)gridDim.x * 8)
      acc += __bfloat162float(dy[row * ld + c]);
  __shared__ float s[8][32];
  s[r][c] = acc;
  __syncthreads();
  if (r == 0) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += s[i][c];
    partials[blockIdx.x * 32 + c] = t;
  }
}

// db[c] += sum over blocks of partials[block][c], always in the same order
__global__ void __launch_bounds__(256)
colsum_finish_kernel(const float* __restrict__ partials, int nblocks, int C, float* __restrict__ db) {
  pdl_sync();
  const int c = threadIdx.x & 31, r = threadIdx.x >> 5;
  float acc = 0.f;
  for (int b = r; b < nblocks; b += 8) acc += partials[b * 32 + c];
  __shared__ float s[8][32];
  s[r][c] = acc;
  __syncthreads();
  if (r == 0 && c < C) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += s[i][c];
    db[c] += t;
  }
}

}  // namespace b200seg

using namespace b200seg;

#define RET_LAUNCH()                        \
  do {                                      \
    cudaError_t e_ = cudaGetLastError();    \
    return e_ == cudaSuccess ? 0 : (int)e_; \
  } while (0)

static inline int pix_blocks(long long P) {
  long long b = (P + 255) / 256;
  return (int)(b < 1 ? 1 : (b > 296 ? 296 : b));
}

extern "C" int32_t b200seg_spatial_softmax_blocks(int32_t P) { return pix_blocks(P); }

extern "C" int b200seg_spatial_softmax_fwd(const float* logits, int32_t ld, int32_t n, int32_t P, int32_t K,
                                           float* partial_ws, void* probs_bf16, float* stat_out, void* stream) {
  if (!logits || !partial_ws || !probs_bf16 || K > KP || K < 1) return B200SEG_E_BADARG;
  const int B = pix_blocks(P);
  launch_k(spatial_stats_kernel, dim3(B, n), dim3(256), 0, (cudaStream_t)stream, logits, ld, P, K, partial_ws);
  launch_k(spatial_apply_kernel, dim3(B, n), dim3(256), 0, (cudaStream_t)stream, logits, ld, P, K, partial_ws, B,
                                                                     (__nv_bfloat16*)probs_bf16, stat_out);
  RET_LAUNCH();
}

extern "C" int b200seg_spatial_softmax_bwd(const float* dprobs, int32_t ldd, const void* probs_bf16, int32_t n, int32_t P,
                                           int32_t K, float* partial_ws, void* dlogit_bf16, int32_t accumulate,
                                           void* stream) {
  if (!dprobs || !probs_bf16 || !partial_ws || !dlogit_bf16 || K > KP) return B200SEG_E_BADARG;
  const int B = pix_blocks(P);
  launch_k(spatial_bwd_reduce_kernel, dim3(B, n), dim3(256), 0, (cudaStream_t)stream, dprobs, ldd,
           (const __nv_bfloat16*)probs_bf16, P, K, partial_ws);
  launch_k(spatial_bwd_apply_kernel, dim3(B, n), dim3(256), 0, (cudaStream_t)stream, dprobs, ldd,
           (const __nv_bfloat16*)probs_bf16, P, K, partial_ws, B, (__nv_bfloat16*)dlogit_bf16, accumulate);
  RET_LAUNCH();
}

extern "C" int b200seg_class_softmax_fwd(const float* x, int32_t ld, int64_t P, int32_t K, float scale, void* sim_bf16,
                                         void* stream) {
  if (!x || !sim_bf16 || K > KP) return B200SEG_E_BADARG;
  launch_k(class_softmax_fwd_kernel, dim3(pix_blocks(P) * 4), dim3(256), 0, (cudaStream_t)stream, x, ld, P, K, scale,
                                                                                (__nv_bfloat16*)sim_bf16);
  RET_LAUNCH();
}

extern "C" int b200seg_class_softmax_bwd(const float* dsim, int32_t ld, const void* sim_bf16, int64_t P, int32_t K,
                                         float scale, void* ds_bf16, void* stream) {
  if (!dsim || !sim_bf16 || !ds_bf16 || K > KP) return B200SEG_E_BADARG;
  launch_k(class_softmax_bwd_kernel, dim3(pix_blocks(P) * 4), dim3(256), 0, (cudaStream_t)stream, dsim, ld,
           (const __nv_bfloat16*)sim_bf16, P, K, scale, (__nv_bfloat16*)ds_bf16);
  RET_LAUNCH();
}

extern "C" int b200seg_transpose_pad(const void* src, int32_t src_fp32, int32_t R, int32_t C, int32_t ld, void* dst_bf16,
                                     int32_t rpad, void* stream) {
  if (!src || !dst_bf16 || rpad < R) return B200SEG_E_BADARG;
  launch_k(transpose_pad_kernel, dim3((C * rpad + 255) / 256), dim3(256), 0, (cudaStream_t)stream, src, src_fp32, R,
           C, ld, (__nv_bfloat16*)dst_bf16, rpad);
  RET_LAUNCH();
}

extern "C" int b200seg_cast_rows(const float* src, int32_t src_ld, void* dst_bf16, int32_t dst_ld, int64_t rows,
                                 int32_t C, int32_t accumulate, void* stream) {
  if (!src || !dst_bf16) return B200SEG_E_BADARG;
  long long total = rows * C;
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  launch_k(cast_rows_kernel, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, src, src_ld, (__nv_bfloat16*)dst_bf16,
           dst_ld, rows, C, accumulate);
  RET_LAUNCH();
}

extern "C" int32_t b200seg_bias_grad_blocks(int64_t rows) {
  const long long b = (rows + 7) / 8;
  return (int32_t)(b < 1 ? 1 : (b > 148 * 4 ? 148 * 4 : b));
}

extern "C" int b200seg_bias_grad(const void* dy_bf16, int32_t ld, int64_t rows, int32_t C, float* partials, float* db,
                                 void* stream) {
  if (!dy_bf16 || !partials || !db || C > 32) return B200SEG_E_BADARG;
  const int b = b200seg_bias_grad_blocks(rows);
  launch_k(colsum_kernel, dim3(b), dim3(256), 0, (cudaStream_t)stream, (const __nv_bfloat16*)dy_bf16, ld, rows,
           C, partials);
  launch_k(colsum_finish_kernel, dim3(1), dim3(256), 0, (cudaStream_t)stream, (const float*)partials, b, C, db);
  RET_LAUNCH();
}
