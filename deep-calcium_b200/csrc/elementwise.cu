// Memory-bound kernels of the UNet2DS path: BatchNorm statistics / apply / backward,
// 2x2 max-pool fwd+bwd, dropout, the softmax head fused with loss + metrics + gradient,
// the 8x dihedral test-time augmentation, Keras-form Adam.
// Reference sites: unet_2d_summary.py:154-222 (layers), :585-595 (TTA), utils/neurons.py:13-137
// (losses, metrics, TTA table); Keras 2.0.6 semantics as listed in SURVEY.md section 3.5.
#include <cstdlib>
#include "elementwise.cuh"

namespace dcb {

static inline int ew_grid(long long work_items, int block) {
  long long g = (work_items + block - 1) / block;
  long long cap = (long long)sm_count() * 16;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

// ---------------------------------------------------------------- cast
template <typename T>
__global__ void cast_f32_kernel(const float* __restrict__ in, long long n, T* __restrict__ out) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = from_f32<T>(in[i]);
}
template <typename T>
__global__ void cast_to_f32_kernel(const T* __restrict__ in, long long n, float* __restrict__ out) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = to_f32<T>(in[i]);
}

// ---------------------------------------------------------------- BN (inference fold)
__global__ void bn_fold_kernel(const float* gamma, const float* beta, const float* mean, const float* var,
                               const float* bias, int C, float eps, float* scale, float* shift) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float s = gamma[c] * rsqrtf(var[c] + eps);
  scale[c] = s;
  shift[c] = beta[c] + ((bias ? bias[c] : 0.f) - mean[c]) * s;
}

// ---------------------------------------------------------------- BN batch statistics
// x [M][C]; each thread owns 8 consecutive channels (one 16-byte bf16 load); the CTA walks a contiguous
// row range with 4 independent row loads in flight per thread.
template <typename T, int VEC>
__global__ void __launch_bounds__(256)
bn_stats_kernel(const T* __restrict__ x, long long M, int C, double* __restrict__ sums) {
  const int lanes_c = C / VEC;                // threads per row
  const int rows_par = 256 / lanes_c;         // rows processed in parallel by the CTA
  const int tc = threadIdx.x % lanes_c, tr = threadIdx.x / lanes_c;
  const long long rows_per_cta = (M + gridDim.x - 1) / gridDim.x;
  const long long r0 = (long long)blockIdx.x * rows_per_cta;
  long long r1 = r0 + rows_per_cta; if (r1 > M) r1 = M;
  float s[VEC], q[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) { s[i] = 0.f; q[i] = 0.f; }
  const T* base = x + tc * VEC;
  long long r = r0 + tr;
  for (; r + 3LL * rows_par < r1; r += 4LL * rows_par) {
    float v[4][VEC];
#pragma unroll
    for (int u = 0; u < 4; ++u) loadv<T, VEC>(base + (r + (long long)u * rows_par) * C, v[u]);
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int i = 0; i < VEC; ++i) { s[i] += v[u][i]; q[i] = fmaf(v[u][i], v[u][i], q[i]); }
  }
  for (; r < r1; r += rows_par) {
    float v[VEC];
    loadv<T, VEC>(base + r * C, v);
#pragma unroll
    for (int i = 0; i < VEC; ++i) { s[i] += v[i]; q[i] = fmaf(v[i], v[i], q[i]); }
  }
  __shared__ float sh[256 * 2 * VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) { sh[threadIdx.x * 2 * VEC + i] = s[i]; sh[threadIdx.x * 2 * VEC + VEC + i] = q[i]; }
  __syncthreads();
  // (channel-lane, component) pairs; sum over the row-parallel copies, one fp64 atomic per channel and CTA
  for (int idx = threadIdx.x; idx < lanes_c * 2 * VEC; idx += 256) {
    const int lc = idx / (2 * VEC), comp = idx % (2 * VEC);
    double acc = 0;
    for (int rr = 0; rr < rows_par; ++rr) acc += (double)sh[(rr * lanes_c + lc) * 2 * VEC + comp];
    atomicAdd(&sums[(comp / VEC) * C + lc * VEC + (comp % VEC)], acc);
  }
}

__global__ void bn_finalize_kernel(const double* __restrict__ sums, long long M, int C, const float* gamma,
                                   const float* beta, float eps, float momentum, float* moving_mean,
                                   float* moving_var, float* scale, float* shift, float* mean_out, float* rstd_out) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double mean = sums[c] / (double)M;
  double var = sums[C + c] / (double)M - mean * mean;
  if (var < 0) var = 0;
  const float rstd = (float)(1.0 / sqrt(var + (double)eps));
  const float sc = gamma[c] * rstd;
  scale[c] = sc;
  shift[c] = beta[c] - (float)mean * sc;
  mean_out[c] = (float)mean;
  rstd_out[c] = rstd;
  if (moving_mean) {   // Keras: moving <- moving*m + batch*(1-m), biased batch variance
    moving_mean[c] = moving_mean[c] * momentum + (float)mean * (1.f - momentum);
    moving_var[c] = moving_var[c] * momentum + (float)var * (1.f - momentum);
  }
}

// y = relu(x*scale + shift) [* dropout keep-scale]; per-channel coefficients staged in shared memory,
// VEC (4 or 8) channels per thread and iteration
template <typename T, int VEC>
__global__ void __launch_bounds__(256)
bn_apply_kernel(const T* __restrict__ x, long long M, int C, const float* __restrict__ scale,
                const float* __restrict__ shift, int relu, float p_drop, unsigned long long seed,
                const unsigned long long* __restrict__ seed_dev, uint32_t layer, T* __restrict__ y) {
  extern __shared__ float s_coef[];
  float* s_sc = s_coef; float* s_sh = s_coef + C;
  for (int c = threadIdx.x; c < C; c += blockDim.x) { s_sc[c] = scale[c]; s_sh[c] = shift[c]; }
  __syncthreads();
  if (seed_dev) seed ^= *seed_dev;
  const long long nv = M * C / VEC;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)((i * VEC) % C);
    float v[VEC];
    loadv<T, VEC>(x + i * VEC, v);
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      v[j] = fmaf(v[j], s_sc[c + j], s_sh[c + j]);
      if (relu) v[j] = fmaxf(v[j], 0.f);
    }
    if (p_drop > 0.f) {
#pragma unroll
      for (int h = 0; h < VEC / 4; ++h) {
        const float4 k = dropout_scale4(seed, layer, (unsigned long long)(i * (VEC / 4) + h), p_drop);
        v[4 * h] *= k.x; v[4 * h + 1] *= k.y; v[4 * h + 2] *= k.z; v[4 * h + 3] *= k.w;
      }
    }
    storev<T, VEC>(y + i * VEC, v);
  }
}

// Training forward in one pass over the data: every CTA derives the per-channel scale / shift from the batch sums in
// its prologue (C <= 2048 channels: a few microseconds of fp64 per CTA instead of a separate launch per layer);
// block 0 also publishes scale / shift / mean / rstd for the backward pass and updates the moving statistics.
template <typename T, int VEC>
__global__ void __launch_bounds__(256)
bn_finalize_apply_kernel(const T* __restrict__ x, long long M, int C, const double* __restrict__ sums, long long M_total,
                         const float* __restrict__ gamma, const float* __restrict__ beta, float eps, float momentum,
                         float* moving_mean, float* moving_var, float* scale_out, float* shift_out, float* mean_out,
                         float* rstd_out, int relu, float p_drop, unsigned long long seed,
                         const unsigned long long* __restrict__ seed_dev, uint32_t layer, T* __restrict__ y) {
  extern __shared__ float s_coef[];
  float* s_sc = s_coef; float* s_sh = s_coef + C;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const double mean = sums[c] / (double)M_total;
    double var = sums[C + c] / (double)M_total - mean * mean;
    if (var < 0) var = 0;
    const float rstd = (float)(1.0 / sqrt(var + (double)eps));
    const float sc = gamma[c] * rstd;
    const float sh = beta[c] - (float)mean * sc;
    s_sc[c] = sc; s_sh[c] = sh;
    if (blockIdx.x == 0) {
      scale_out[c] = sc; shift_out[c] = sh; mean_out[c] = (float)mean; rstd_out[c] = rstd;
      if (moving_mean) {   // Keras: moving <- moving*m + batch*(1-m), biased batch variance
        moving_mean[c] = moving_mean[c] * momentum + (float)mean * (1.f - momentum);
        moving_var[c] = moving_var[c] * momentum + (float)var * (1.f - momentum);
      }
    }
  }
  __syncthreads();
  if (seed_dev) seed ^= *seed_dev;
  const long long nv = M * C / VEC;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)((i * VEC) % C);
    float v[VEC];
    loadv<T, VEC>(x + i * VEC, v);
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      v[j] = fmaf(v[j], s_sc[c + j], s_sh[c + j]);
      if (relu) v[j] = fmaxf(v[j], 0.f);
    }
    if (p_drop > 0.f) {
#pragma unroll
      for (int h = 0; h < VEC / 4; ++h) {
        const float4 k = dropout_scale4(seed, layer, (unsigned long long)(i * (VEC / 4) + h), p_drop);
        v[4 * h] *= k.x; v[4 * h + 1] *= k.y; v[4 * h + 2] *= k.z; v[4 * h + 3] *= k.w;
      }
    }
    storev<T, VEC>(y + i * VEC, v);
  }
}

// ---------------------------------------------------------------- BN + ReLU (+dropout) backward
// dz = dY * keepscale * [x*scale+shift > 0];  sums[c] += dz ; sums[C+c] += dz * xhat, xhat = (x-mean)*rstd
// 8 channels per thread, 2 independent rows in flight.
template <typename T, int VEC>
__global__ void __launch_bounds__(256)
bn_bwd_reduce_kernel(const float* __restrict__ dy, int ldy, int offy, const T* __restrict__ x, long long M, int C,
                     const float* __restrict__ scale, const float* __restrict__ shift,
                     const float* __restrict__ mean, const float* __restrict__ rstd, float p_drop,
                     unsigned long long seed, const unsigned long long* __restrict__ seed_dev, uint32_t layer,
                     double* __restrict__ sums) {
  if (seed_dev) seed ^= *seed_dev;
  const int lanes_c = C / VEC;
  const int rows_par = 256 / lanes_c;
  const int tc = threadIdx.x % lanes_c, tr = threadIdx.x / lanes_c;
  const long long rows_per_cta = (M + gridDim.x - 1) / gridDim.x;
  const long long r0 = (long long)blockIdx.x * rows_per_cta;
  long long r1 = r0 + rows_per_cta; if (r1 > M) r1 = M;
  const int c = tc * VEC;
  float sc[VEC], sh[VEC], mu[VEC], rs[VEC], s[VEC], q[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) { sc[i] = scale[c + i]; sh[i] = shift[c + i]; mu[i] = mean[c + i]; rs[i] = rstd[c + i]; s[i] = 0.f; q[i] = 0.f; }
  auto accumulate = [&](long long r, const float (&g8)[VEC], const float (&v)[VEC]) {
    float g[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) g[i] = g8[i];
    if (p_drop > 0.f) {
      const unsigned long long i4 = (unsigned long long)((r * C + c) >> 2);
      const float4 k0 = dropout_scale4(seed, layer, i4, p_drop);
      g[0] *= k0.x; g[1] *= k0.y; g[2] *= k0.z; g[3] *= k0.w;
      if constexpr (VEC == 8) {
        const float4 k1 = dropout_scale4(seed, layer, i4 + 1, p_drop);
        g[4] *= k1.x; g[5] *= k1.y; g[6] *= k1.z; g[7] *= k1.w;
      }
    }
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      if (fmaf(v[i], sc[i], sh[i]) <= 0.f) g[i] = 0.f;
      s[i] += g[i];
      q[i] = fmaf(g[i], (v[i] - mu[i]) * rs[i], q[i]);
    }
  };
  long long r = r0 + tr;
  for (; r + rows_par < r1; r += 2LL * rows_par) {
    float g0[VEC], g1[VEC], v0[VEC], v1[VEC];
    loadv<float, VEC>(dy + r * ldy + offy + c, g0);
    loadv<float, VEC>(dy + (r + rows_par) * ldy + offy + c, g1);
    loadv<T, VEC>(x + r * C + c, v0);
    loadv<T, VEC>(x + (r + rows_par) * C + c, v1);
    accumulate(r, g0, v0);
    accumulate(r + rows_par, g1, v1);
  }
  for (; r < r1; r += rows_par) {
    float g0[VEC], v0[VEC];
    loadv<float, VEC>(dy + r * ldy + offy + c, g0);
    loadv<T, VEC>(x + r * C + c, v0);
    accumulate(r, g0, v0);
  }
  __shared__ float shm[256 * 2 * VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) { shm[threadIdx.x * 2 * VEC + i] = s[i]; shm[threadIdx.x * 2 * VEC + VEC + i] = q[i]; }
  __syncthreads();
  for (int idx = threadIdx.x; idx < lanes_c * 2 * VEC; idx += 256) {
    const int lc = idx / (2 * VEC), comp = idx % (2 * VEC);
    double acc = 0;
    for (int rr = 0; rr < rows_par; ++rr) acc += (double)shm[(rr * lanes_c + lc) * 2 * VEC + comp];
    atomicAdd(&sums[(comp / VEC) * C + lc * VEC + (comp % VEC)], acc);
  }
}

// d_raw = scale * (dz - mean(dz) - xhat * mean(dz*xhat)) = scale*dz + k1*(x - mean) + k0 with per-channel
//   k1 = -scale*rstd*mean(dz*xhat),  k0 = -scale*mean(dz)                    (fp64 once per CTA, then fp32 FMAs)
// block 0 also emits dgamma/dbeta
template <typename T, int VEC>
__global__ void __launch_bounds__(256)
bn_bwd_apply_kernel(const float* __restrict__ dy, int ldy, int offy, const T* __restrict__ x, long long M,
                    int C, const float* __restrict__ scale, const float* __restrict__ shift,
                    const float* __restrict__ mean, const float* __restrict__ rstd, float p_drop,
                    unsigned long long seed, const unsigned long long* __restrict__ seed_dev,
                    uint32_t layer, const double* __restrict__ sums, long long M_total,
                    float dgb_scale, T* __restrict__ draw, float* __restrict__ dgamma,
                    float* __restrict__ dbeta) {
  extern __shared__ float s_coef[];
  float* s_sc = s_coef; float* s_sh = s_coef + C; float* s_k1 = s_coef + 2 * C; float* s_k0 = s_coef + 3 * C;
  float* s_mu = s_coef + 4 * C;
  const double invM = 1.0 / (double)M_total;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const double sc = scale[c], m1 = sums[c] * invM, m2 = sums[C + c] * invM;
    const double k1 = -sc * (double)rstd[c] * m2;
    s_sc[c] = scale[c]; s_sh[c] = shift[c];
    s_k1[c] = (float)k1;
    s_k0[c] = (float)(-sc * m1);
    s_mu[c] = mean[c];
    if (blockIdx.x == 0) {
      if (dbeta) dbeta[c] = (float)(sums[c] * (double)dgb_scale);
      if (dgamma) dgamma[c] = (float)(sums[C + c] * (double)dgb_scale);
    }
  }
  __syncthreads();
  if (seed_dev) seed ^= *seed_dev;
  const int cvn = C / VEC;
  const long long nv = M * cvn;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cvn;
    const int c = (int)(i % cvn) * VEC;
    float g[VEC], v[VEC];
    loadv<float, VEC>(dy + r * ldy + offy + c, g);
    loadv<T, VEC>(x + r * C + c, v);
    if (p_drop > 0.f) {
#pragma unroll
      for (int h = 0; h < VEC / 4; ++h) {
        const float4 k = dropout_scale4(seed, layer, (unsigned long long)(i * (VEC / 4) + h), p_drop);
        g[4 * h] *= k.x; g[4 * h + 1] *= k.y; g[4 * h + 2] *= k.z; g[4 * h + 3] *= k.w;
      }
    }
    float o[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      const float gz = fmaf(v[j], s_sc[c + j], s_sh[c + j]) <= 0.f ? 0.f : g[j];
      o[j] = fmaf(s_sc[c + j], gz, fmaf(s_k1[c + j], v[j] - s_mu[c + j], s_k0[c + j]));
    }
    storev<T, VEC>(draw + r * C + c, o);
  }
}

// ---------------------------------------------------------------- training crop sampler (device half)
// The reference's _batch_gen (unet_2d_summary.py:434-530) draws, per crop, a dataset, a neuron-centred window with
// jitter and a random sequence of flips / rot90s with the global numpy RNG, then slices, zero-fills and transforms the
// window in a Python loop.  Here the host keeps the RNG stream (a handful of integers per crop) and the device does the
// pixel work: desc[b] = {dataset, y0, x0, valid rows, valid cols, m00, m01, m10, m11, t0, t1, 0}; output pixel (i, j)
// of crop b reads window position (wi, wj) = (m00*i + m01*j + t0, m10*i + m11*j + t1) - the composition of the
// crop's flips / rotations as one affine index map on the square window - and is 0 outside the valid part.
__global__ void crop_batch_kernel(const long long* __restrict__ img_ptrs, const long long* __restrict__ mask_ptrs,
                                  const int* __restrict__ widths, const int* __restrict__ desc, int B, int n,
                                  float* __restrict__ xo, uint8_t* __restrict__ yo) {
  const long long total = (long long)B * n * n;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(idx % n), i = (int)((idx / n) % n), b = (int)(idx / ((long long)n * n));
    const int* d = desc + 12 * b;
    const int wi = d[5] * i + d[6] * j + d[9], wj = d[7] * i + d[8] * j + d[10];
    float v = 0.f; uint8_t m = 0;
    if (wi >= 0 && wi < d[3] && wj >= 0 && wj < d[4]) {
      const long long off = (long long)(d[1] + wi) * widths[d[0]] + (d[2] + wj);
      v = reinterpret_cast<const float*>(img_ptrs[d[0]])[off];
      m = reinterpret_cast<const uint8_t*>(mask_ptrs[d[0]])[off];
    }
    xo[idx] = v; yo[idx] = m;
  }
}

// ---------------------------------------------------------------- nearest 2x upsampling (+dropout)
// UpSampling2D of the non-default `upsampling_or_transpose='upsampling'` graph (unet_2d_summary.py:160-161), followed by
// the Dropout that the reference applies to the upsampled tensor (:198-216).  y[n][2h+a][2w+b][c] = x[n][h][w][c] * keep.
template <typename T>
__global__ void upsample2x_kernel(const T* __restrict__ x, int N, int h, int w, int C, float p_drop, unsigned long long seed,
                                  const unsigned long long* __restrict__ seed_dev, uint32_t layer, T* __restrict__ y) {
  if (seed_dev) seed ^= *seed_dev;
  const int c4n = C >> 2;
  const long long n4 = (long long)N * (2 * h) * (2 * w) * c4n;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % c4n) * 4;
    long long r = i / c4n;
    const int ox = (int)(r % (2 * w)); r /= 2 * w;
    const int oy = (int)(r % (2 * h)); const int n = (int)(r / (2 * h));
    float4 v = load4<T>(x + (((long long)n * h + (oy >> 1)) * w + (ox >> 1)) * C + c);
    if (p_drop > 0.f) {
      const float4 k = dropout_scale4(seed, layer, (unsigned long long)i, p_drop);
      v.x *= k.x; v.y *= k.y; v.z *= k.z; v.w *= k.w;
    }
    store4<T>(y + i * 4, v);
  }
}

// dx[n][h][w][c] = sum over the 2x2 block of dy[n][2h+a][2w+b][offy + c] * keep   (dy fp32 view, dx fp32)
__global__ void upsample2x_bwd_kernel(const float* __restrict__ dy, int ldy, int offy, int N, int h, int w, int C, float p_drop,
                                      unsigned long long seed, const unsigned long long* __restrict__ seed_dev, uint32_t layer,
                                      float* __restrict__ dx) {
  if (seed_dev) seed ^= *seed_dev;
  const int c4n = C >> 2;
  const long long n4 = (long long)N * h * w * c4n;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % c4n) * 4;
    long long r = i / c4n;
    const int ix = (int)(r % w); r /= w;
    const int iy = (int)(r % h); const int n = (int)(r / h);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int b = 0; b < 2; ++b) {
        const long long opix = ((long long)n * (2 * h) + (2 * iy + a)) * (2 * w) + (2 * ix + b);
        float4 g = load4<float>(dy + opix * ldy + offy + c);
        if (p_drop > 0.f) {   // same counter as the forward: flat index of the upsampled element / 4
          const float4 k = dropout_scale4(seed, layer, (unsigned long long)(opix * c4n + (c >> 2)), p_drop);
          g.x *= k.x; g.y *= k.y; g.z *= k.z; g.w *= k.w;
        }
        acc.x += g.x; acc.y += g.y; acc.z += g.z; acc.w += g.w;
      }
    *reinterpret_cast<float4*>(dx + i * 4) = acc;
  }
}

// ---------------------------------------------------------------- 2x2 max-pool
// 8 channels (16 B of bf16) per thread: the four window loads are independent 16-byte requests
template <typename T>
__global__ void __launch_bounds__(256)
maxpool2x2_v8_kernel(const T* __restrict__ x, int N, int H, int W, int C, T* __restrict__ y) {
  const int OH = H / 2, OW = W / 2, c8n = C >> 3;
  const long long n8 = (long long)N * OH * OW * c8n;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    long long t = i;
    const int c = (int)(t % c8n) * 8; t /= c8n;
    const int ow = (int)(t % OW); t /= OW;
    const int oh = (int)(t % OH); const int n = (int)(t / OH);
    const T* p = x + (((long long)n * H + 2 * oh) * W + 2 * ow) * C + c;
    float a[8], b[8], d[8], e[8], m[8];
    load8<T>(p, a); load8<T>(p + C, b); load8<T>(p + (long long)W * C, d); load8<T>(p + (long long)W * C + C, e);
#pragma unroll
    for (int q = 0; q < 8; ++q) m[q] = fmaxf(fmaxf(a[q], b[q]), fmaxf(d[q], e[q]));
    store8<T>(y + i * 8, m);
  }
}

template <typename T>
__global__ void maxpool2x2_kernel(const T* __restrict__ x, int N, int H, int W, int C, T* __restrict__ y) {
  const int OH = H / 2, OW = W / 2, c4n = C >> 2;
  const long long n4 = (long long)N * OH * OW * c4n;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    long long t = i;
    const int c = (int)(t % c4n) * 4; t /= c4n;
    const int ow = (int)(t % OW); t /= OW;
    const int oh = (int)(t % OH); const int n = (int)(t / OH);
    const T* p = x + (((long long)n * H + 2 * oh) * W + 2 * ow) * C + c;
    const float4 a = load4<T>(p), b = load4<T>(p + C), d = load4<T>(p + (long long)W * C), e = load4<T>(p + (long long)W * C + C);
    float4 m;
    m.x = fmaxf(fmaxf(a.x, b.x), fmaxf(d.x, e.x)); m.y = fmaxf(fmaxf(a.y, b.y), fmaxf(d.y, e.y));
    m.z = fmaxf(fmaxf(a.z, b.z), fmaxf(d.z, e.z)); m.w = fmaxf(fmaxf(a.w, b.w), fmaxf(d.w, e.w));
    store4<T>(y + i * 4, m);
  }
}

// out[n,h,w,c] = skipgrad[n,h,w, off+c] + (first position in the 2x2 window whose y equals the pooled max ? dpool : 0)
template <typename T>
__global__ void pool_bwd_add_kernel(const float* __restrict__ skipgrad, int lds, int offs, const T* __restrict__ y,
                                    const T* __restrict__ pooled, const float* __restrict__ dpool, int N, int H, int W,
                                    int C, float* __restrict__ out) {
  const int OH = H / 2, OW = W / 2, c4n = C >> 2;
  const long long n4 = (long long)N * OH * OW * c4n;
  if (threadIdx.x == 0) pdl_trigger();
  pdl_wait();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    long long t = i;
    const int c = (int)(t % c4n) * 4; t /= c4n;
    const int ow = (int)(t % OW); t /= OW;
    const int oh = (int)(t % OH); const int n = (int)(t / OH);
    const float4 pm = load4<T>(pooled + i * 4);
    const float4 dp = load4<float>(dpool + i * 4);
    bool done[4] = {false, false, false, false};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const long long pix = ((long long)n * H + 2 * oh + (q >> 1)) * W + 2 * ow + (q & 1);
      const float4 v = load4<T>(y + pix * C + c);
      float4 g = skipgrad ? load4<float>(skipgrad + pix * lds + offs + c) : make_float4(0.f, 0.f, 0.f, 0.f);
      if (!done[0] && v.x == pm.x) { g.x += dp.x; done[0] = true; }
      if (!done[1] && v.y == pm.y) { g.y += dp.y; done[1] = true; }
      if (!done[2] && v.z == pm.z) { g.z += dp.z; done[2] = true; }
      if (!done[3] && v.w == pm.w) { g.w += dp.w; done[3] = true; }
      store4<float>(out + pix * C + c, g);
    }
  }
}

// ---------------------------------------------------------------- head: 1x1 conv C->2 + softmax[...,-1]
// (unet_2d_summary.py:221-222)  p = softmax(z)[1] = sigmoid(z1 - z0)
template <typename T>
__device__ __forceinline__ float head_logit(const T* __restrict__ row, int C, const float* wd, float bd) {
  float acc = bd;
  for (int c = 0; c < C; c += 4) {
    const float4 v = load4<T>(row + c);
    acc = fmaf(v.x, wd[c], acc); acc = fmaf(v.y, wd[c + 1], acc);
    acc = fmaf(v.z, wd[c + 2], acc); acc = fmaf(v.w, wd[c + 3], acc);
  }
  return acc;
}

template <typename T>
__global__ void __launch_bounds__(256)
head_fwd_kernel(const T* __restrict__ x, long long M, int C, const float* __restrict__ w, const float* __restrict__ b,
                float* __restrict__ logit, float* __restrict__ prob) {
  __shared__ float wd[512];
  for (int c = threadIdx.x; c < C; c += blockDim.x) wd[c] = w[c * 2 + 1] - w[c * 2];
  __syncthreads();
  const float bd = b[1] - b[0];
  for (long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x; m < M; m += (long long)gridDim.x * blockDim.x) {
    const float z = head_logit<T>(x + m * C, C, wd, bd);
    if (logit) logit[m] = z;
    if (prob) prob[m] = 1.f / (1.f + __expf(-z));
  }
}

// sums: [0]=sum yt  [1]=sum p  [2]=sum yt*p  [3]=sum p^2  [4]=sum round(p)  [5]=sum yt*round(p)
//       [6]=sum BCE terms (Keras clip 1e-7)  [7]=sum weighted-BCE terms (utils/neurons.py:13-29)
template <typename T>
__global__ void __launch_bounds__(256)
head_loss_fwd_kernel(const T* __restrict__ x, long long M, int C, const float* __restrict__ w,
                     const float* __restrict__ b, const uint8_t* __restrict__ yt, float* __restrict__ prob,
                     double* __restrict__ sums) {
  __shared__ float wd[512];
  __shared__ double red[8][8];
  for (int c = threadIdx.x; c < C; c += blockDim.x) wd[c] = w[c * 2 + 1] - w[c * 2];
  __syncthreads();
  const float bd = b[1] - b[0];
  float s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x; m < M; m += (long long)gridDim.x * blockDim.x) {
    const float z = head_logit<T>(x + m * C, C, wd, bd);
    const float p = 1.f / (1.f + expf(-z));
    prob[m] = p;
    const float t = (float)yt[m];
    const float rp = rintf(p);   // K.round = round half to even
    s[0] += t; s[1] += p; s[2] += t * p; s[3] += p * p; s[4] += rp; s[5] += t * rp;
    const float pc = fminf(fmaxf(p, 1e-7f), 1.f - 1e-7f);
    s[6] += -(t * logf(pc) + (1.f - t) * logf(1.f - pc));
    s[7] += -(2.f * t * logf(p + 1e-7f) + (1.f - t) * logf(1.f - p + 1e-7f));
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const double v = warp_sum((double)s[i]);
    if (lane == 0) red[i][warp] = v;
  }
  __syncthreads();
  if (threadIdx.x < 8) {
    double acc = 0;
    for (int wv = 0; wv < 8; ++wv) acc += red[threadIdx.x][wv];
    atomicAdd(&sums[threadIdx.x], acc);
  }
}

__device__ __forceinline__ float loss_grad_wrt_p(int loss, float p, float t, const double* sums, double invM) {
  switch (loss) {
    case DCB_LOSS_DICE: {        // utils/neurons.py:78-83
      const double I = sums[2], D = sums[0] + sums[1] + 1e-7;
      return (float)(-2.0 * ((double)t * D - I) / (D * D));
    }
    case DCB_LOSS_DICESQ: {      // utils/neurons.py:86-94 (yt in {0,1} so yt^2 = yt)
      const double I = sums[2], Q = sums[0] + sums[3] + 1e-7;
      return (float)(-2.0 * ((double)t * Q - I * 2.0 * (double)p) / (Q * Q));
    }
    case DCB_LOSS_BCE: {
      if (p <= 1e-7f || p >= 1.f - 1e-7f) return 0.f;
      return (float)invM * (-t / p + (1.f - t) / (1.f - p));
    }
    default:                     // weighted BCE, weightpos=2, weightneg=1
      return (float)invM * (-2.f * t / (p + 1e-7f) + (1.f - t) / (1.f - p + 1e-7f));
  }
}

// dx[m][c] = dz1 * (w[c][1]-w[c][0]),  dz1 = p(1-p) dL/dp ;  dwb[c*2+j] accumulates head kernel grads,
// dwb[2C + j] the bias grads (double atomics)
template <typename T>
__global__ void __launch_bounds__(256)
head_loss_bwd_kernel(const T* __restrict__ x, long long M, int C, const float* __restrict__ w,
                     const uint8_t* __restrict__ yt, const float* __restrict__ prob, const double* __restrict__ sums,
                     int loss, long long M_total, float* __restrict__ dx, double* __restrict__ dwb) {
  __shared__ float wd[512];
  __shared__ float accw[512];
  __shared__ float accb;
  for (int c = threadIdx.x; c < C; c += blockDim.x) { wd[c] = w[c * 2 + 1] - w[c * 2]; accw[c] = 0.f; }
  if (threadIdx.x == 0) accb = 0.f;
  __syncthreads();
  const double invM = 1.0 / (double)M_total;
  const int lane = threadIdx.x & 31;
  float myw[16];                 // lane l owns channels l, l+32, ... (C <= 512)
#pragma unroll
  for (int i = 0; i < 16; ++i) myw[i] = 0.f;
  float myb = 0.f;
  // block-uniform trip count so that the warp shuffles below are convergent
  for (long long base = (long long)blockIdx.x * blockDim.x; base < M; base += (long long)gridDim.x * blockDim.x) {
    const long long m = base + threadIdx.x;
    const bool valid = m < M;
    float dz1 = 0.f;
    if (valid) {
      const float p = prob[m];
      const float g = loss_grad_wrt_p(loss, p, (float)yt[m], sums, invM);
      dz1 = p * (1.f - p) * g;
    }
    myb += dz1;
    for (int c = 0; c < C; c += 4) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (valid) {
        v = load4<T>(x + m * C + c);
        store4<float>(dx + m * C + c, make_float4(dz1 * wd[c], dz1 * wd[c + 1], dz1 * wd[c + 2], dz1 * wd[c + 3]));
      }
      const float r0 = warp_sum(v.x * dz1), r1 = warp_sum(v.y * dz1), r2 = warp_sum(v.z * dz1), r3 = warp_sum(v.w * dz1);
      const int slot = c >> 5, l0 = c & 31;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        if (i == slot) {
          if (lane == l0) myw[i] += r0;
          if (lane == l0 + 1) myw[i] += r1;
          if (lane == l0 + 2) myw[i] += r2;
          if (lane == l0 + 3) myw[i] += r3;
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const int c = i * 32 + lane;
    if (c < C) atomicAdd(&accw[c], myw[i]);
  }
  myb = warp_sum(myb);
  if (lane == 0) atomicAdd(&accb, myb);
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    atomicAdd(&dwb[c * 2 + 1], (double)accw[c]);
    atomicAdd(&dwb[c * 2], -(double)accw[c]);
  }
  if (threadIdx.x == 0) { atomicAdd(&dwb[2 * C + 1], (double)accb); atomicAdd(&dwb[2 * C], -(double)accb); }
}

// Same contract for C == 32 (nb_filters_base = 32, the benchmarked model): every thread keeps its own 32 partial kernel
// gradients in registers over all its pixels and the CTA reduces them ONCE through shared memory - the generic kernel
// above pays 32 warp reductions (160 shuffles) per 32 pixels inside the loop (48 us of the 32-crop step).
template <typename T>
__global__ void __launch_bounds__(256)
head_loss_bwd_c32_kernel(const T* __restrict__ x, long long M, const float* __restrict__ w, const uint8_t* __restrict__ yt,
                         const float* __restrict__ prob, const double* __restrict__ sums, int loss, long long M_total,
                         float* __restrict__ dx, double* __restrict__ dwb, float* __restrict__ gpix, float* __restrict__ wd_out) {
  // gpix != null: dL/dx is the rank-1 product gpix[m] * wd[c] - only its two factors are written (4 bytes per pixel instead of
  // 128), the BatchNorm backward of the last block rebuilds it on the fly (dcb_bn_train_bwd_rank1)
  constexpr int C = 32;
  __shared__ float wd[C];
  __shared__ float red[8][C + 1];
  if (threadIdx.x < C) {
    wd[threadIdx.x] = w[threadIdx.x * 2 + 1] - w[threadIdx.x * 2];
    if (wd_out && blockIdx.x == 0) wd_out[threadIdx.x] = wd[threadIdx.x];
  }
  __syncthreads();
  const double invM = 1.0 / (double)M_total;
  float acc[C];
#pragma unroll
  for (int c = 0; c < C; ++c) acc[c] = 0.f;
  float accb = 0.f;
  for (long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x; m < M; m += (long long)gridDim.x * blockDim.x) {
    const float p = prob[m];
    const float g = loss_grad_wrt_p(loss, p, (float)yt[m], sums, invM);
    const float dz1 = p * (1.f - p) * g;
    accb += dz1;
    if (gpix) gpix[m] = dz1;
#pragma unroll
    for (int c = 0; c < C; c += 8) {
      float v[8];
      load8<T>(x + m * C + c, v);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[c + j] = fmaf(v[j], dz1, acc[c + j]);
      if (!gpix) {
        store4<float>(dx + m * C + c, make_float4(dz1 * wd[c], dz1 * wd[c + 1], dz1 * wd[c + 2], dz1 * wd[c + 3]));
        store4<float>(dx + m * C + c + 4, make_float4(dz1 * wd[c + 4], dz1 * wd[c + 5], dz1 * wd[c + 6], dz1 * wd[c + 7]));
      }
    }
  }
  // warp reduction of the 33 partials (once per CTA), then across the 8 warps through shared memory
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int c = 0; c < C; ++c) {
    const float r = warp_sum(acc[c]);
    if (lane == 0) red[warp][c] = r;
  }
  accb = warp_sum(accb);
  if (lane == 0) red[warp][C] = accb;
  __syncthreads();
  if (threadIdx.x <= C) {
    float t = 0.f;
#pragma unroll
    for (int wv = 0; wv < 8; ++wv) t += red[wv][threadIdx.x];
    if (threadIdx.x < C) {
      atomicAdd(&dwb[threadIdx.x * 2 + 1], (double)t);
      atomicAdd(&dwb[threadIdx.x * 2], -(double)t);
    } else {
      atomicAdd(&dwb[2 * C + 1], (double)t);
      atomicAdd(&dwb[2 * C], -(double)t);
    }
  }
}

// loss value + the 7 Keras batch metrics (unet_2d_summary.py:398-399) from the 8 sums -> out[8] floats:
// [0]=loss [1]=F1 [2]=prec [3]=reca [4]=dice [5]=dicesq [6]=posyt [7]=posyp
__global__ void head_metrics_kernel(const double* __restrict__ sums, long long M, int loss, float* __restrict__ out,
                                    const double* __restrict__ dwb, int C, float* __restrict__ dw_out) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    const double eps = 1e-7;
    const double syt = sums[0], sp = sums[1], sytp = sums[2], spp = sums[3], srp = sums[4], sytrp = sums[5];
    double L;
    if (loss == DCB_LOSS_DICE) L = 1.0 - 2.0 * sytp / (syt + sp + 1e-7);
    else if (loss == DCB_LOSS_DICESQ) L = -2.0 * sytp / (syt + spp + eps);
    else if (loss == DCB_LOSS_BCE) L = sums[6] / (double)M;
    else L = sums[7] / (double)M;
    const double prec = sytrp / (srp + eps);
    const double fn = syt - sytrp;                 // sum clip(yt - round(p), 0, 1)
    const double reca = sytrp / (sytrp + fn + eps);
    out[0] = (float)L;
    out[1] = (float)(2 * prec * reca / (prec + reca + eps));
    out[2] = (float)prec; out[3] = (float)reca;
    out[4] = (float)(2.0 * sytrp / (syt + srp + 1e-7));
    out[5] = (float)(2.0 * sytp / (syt + spp + eps));
    out[6] = (float)(syt / ((double)M + eps));
    out[7] = (float)(srp / ((double)M + eps));
  }
  if (dwb && dw_out)
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 2 * C + 2; i += gridDim.x * blockDim.x) dw_out[i] = (float)dwb[i];
}

// ---------------------------------------------------------------- 8x dihedral TTA (utils/neurons.py:112-137)
// source coordinate of output (i,j) for transform k on an S x S image
__device__ __forceinline__ void tta_src(int k, int S, int i, int j, int& si, int& sj) {
  switch (k) {
    case 0: si = i; sj = j; break;                    // identity
    case 1: si = S - 1 - i; sj = j; break;            // vflip
    case 2: si = i; sj = S - 1 - j; break;            // hflip
    case 3: si = j; sj = S - 1 - i; break;            // rot90
    case 4: si = S - 1 - i; sj = S - 1 - j; break;    // rot180
    case 5: si = S - 1 - j; sj = i; break;            // rot270
    case 6: si = j; sj = i; break;                    // rot90 + vflip  = transpose
    default: si = S - 1 - j; sj = S - 1 - i; break;   // rot90 + hflip  = anti-transpose
  }
}
// where transform k put input pixel (i,j): the (a,b) with tta_src(k,a,b) == (i,j)
__device__ __forceinline__ void tta_dst(int k, int S, int i, int j, int& a, int& b) {
  switch (k) {
    case 3: a = S - 1 - j; b = i; break;
    case 5: a = j; b = S - 1 - i; break;
    default: tta_src(k, S, i, j, a, b); break;        // the other six are involutions
  }
}
// Overlap-tile TTA.  The canvas is s [hs][ws] reflect-padded at the bottom and right (unet_2d_summary.py:569-571); a plan
// cuts it into S x S tiles with origins (oy[ty], ox[tx]) over an n_ty x n_tx grid, numbered row-major.  A group is the
// tiles tile_first..tile_first+n_tiles-1.  oy == ox == nullptr is the one-tile plan of the 512^2 window (origin 0).
//
// make_batch: out [n_tiles][count][S][S] = each tile of the group under transforms first..first+count-1.  The canvas is
// never materialised: every pixel is read from s through reflect_index in canvas coordinates.
template <typename T>
__global__ void tile_make_batch_kernel(const float* __restrict__ s, int hs, int ws, int S, const int* __restrict__ oy,
                                       const int* __restrict__ ox, int n_tx, int tile_first, int n_tiles, int first,
                                       int count, T* __restrict__ out) {
  const long long per = (long long)S * S;
  const long long n = (long long)n_tiles * count * per;
  if (threadIdx.x == 0) pdl_trigger();
  pdl_wait();
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(idx % S), i = (int)((idx / S) % S);
    const long long b = idx / per;
    const int kk = (int)(b % count), t = tile_first + (int)(b / count);
    const int y0 = oy ? oy[t / n_tx] : 0, x0 = ox ? ox[t % n_tx] : 0;
    int si, sj;
    tta_src(first + kk, S, i, j, si, sj);
    out[idx] = from_f32<T>(s[(long long)reflect_index(y0 + si, hs) * ws + reflect_index(x0 + sj, ws)]);
  }
}

// combine: probs [n_tiles][n_aug][S][S] -> act / mask [hs][ws] at the image pixels the group's tiles own.  Tile (ty, tx)
// owns canvas rows [cy[ty-1], cy[ty]) and columns [cx[tx-1], cx[tx]) (the first / last tile of a row or column from / to
// the canvas edge; cy == cx == nullptr: the one tile owns everything).  act = sum_k float32(inv_k(p_k) / n_aug) in
// float64, in transform order; mask = act > threshold.  Every pixel has exactly one owner and is written once, so the
// result does not depend on how the tiles are grouped.
__global__ void tile_combine_kernel(const float* __restrict__ probs, int S, int hs, int ws, const int* __restrict__ oy,
                                    const int* __restrict__ ox, const int* __restrict__ cy, const int* __restrict__ cx,
                                    int n_ty, int n_tx, int tile_first, int n_tiles, float threshold, int n_aug,
                                    double* __restrict__ act, uint8_t* __restrict__ mask) {
  const long long per = (long long)S * S;
  const long long n = (long long)n_tiles * per;
  if (threadIdx.x == 0) pdl_trigger();
  pdl_wait();
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(idx % S), i = (int)((idx / S) % S), lt = (int)(idx / per);
    const int t = tile_first + lt, ty = t / n_tx, tx = t % n_tx;
    const int y = (oy ? oy[ty] : 0) + i, x = (ox ? ox[tx] : 0) + j;
    if (y < 0 || y >= hs || x < 0 || x >= ws) continue;
    if (cy && ((ty > 0 && y < cy[ty - 1]) || (ty < n_ty - 1 && y >= cy[ty]))) continue;
    if (cx && ((tx > 0 && x < cx[tx - 1]) || (tx < n_tx - 1 && x >= cx[tx]))) continue;
    const float* p = probs + (long long)lt * n_aug * per;
    double acc = 0.0;
    if (n_aug == 1) {
      acc = (double)p[(long long)i * S + j];
    } else {
      for (int k = 0; k < n_aug; ++k) {
        int a, b;
        tta_dst(k, S, i, j, a, b);
        acc += (double)(p[((long long)k * S + a) * S + b] / (float)n_aug);
      }
    }
    const long long o = (long long)y * ws + x;
    if (act) act[o] = acc;
    mask[o] = acc > (double)threshold ? 1 : 0;
  }
}

// ---------------------------------------------------------------- Keras-form Adam (keras.optimizers.Adam, 2.0.6)
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, long long n, float lr_t, const float* __restrict__ lr_t_dev, float b1,
                            float b2, float eps) {
  if (lr_t_dev) lr_t = *lr_t_dev;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float gi = g[i];
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    p[i] = p[i] - lr_t * mi / (sqrtf(vi) + eps);
  }
}

// device-resident step state so that a captured CUDA graph sees a fresh dropout seed and the
// bias-corrected Adam step size on every replay:  state = {iteration (as u64), seed}, lr_t_out = lr_t
__global__ void step_advance_kernel(unsigned long long* state, float lr, float b1, float b2, float* lr_t_out) {
  const unsigned long long t = state[0] + 1ULL;          // Keras: t = iterations + 1
  state[0] = t;
  unsigned long long z = state[1] + 0x9E3779B97F4A7C15ULL;   // splitmix64 step
  state[1] = z;
  const double lr_t = (double)lr * sqrt(1.0 - pow((double)b2, (double)t)) / (1.0 - pow((double)b1, (double)t));
  *lr_t_out = (float)lr_t;
}

}  // namespace dcb

using namespace dcb;

#define DISPATCH_T(dtype, ...)                                                     \
  if ((dtype) == DCB_F32) { using T = float; __VA_ARGS__ }                         \
  else if ((dtype) == DCB_BF16) { using T = __nv_bfloat16; __VA_ARGS__ }           \
  else if ((dtype) == DCB_F16) { using T = __half; __VA_ARGS__ }                   \
  else return fail(DCB_ERR_INVALID_ARGUMENT, "unknown dtype %d", (int)(dtype));

extern "C" int dcb_cast_from_f32(int dtype, const float* in, long long n, void* out, dcb_stream_t stream) {
  DCB_CHECK_ARG(in && out && n >= 0, "dcb_cast_from_f32: bad arguments");
  if (n == 0) return DCB_OK;
  DISPATCH_T(dtype, cast_f32_kernel<T><<<ew_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(in, n, (T*)out);)
  g_launches += 1;
  DCB_LAUNCH_OK("cast_f32_kernel");
  return DCB_OK;
}

extern "C" int dcb_cast_to_f32(int dtype, const void* in, long long n, float* out, dcb_stream_t stream) {
  DCB_CHECK_ARG(in && out && n >= 0, "dcb_cast_to_f32: bad arguments");
  if (n == 0) return DCB_OK;
  DISPATCH_T(dtype, cast_to_f32_kernel<T><<<ew_grid(n, 256), 256, 0, (cudaStream_t)stream>>>((const T*)in, n, out);)
  g_launches += 1;
  DCB_LAUNCH_OK("cast_to_f32_kernel");
  return DCB_OK;
}

extern "C" int dcb_bn_fold(const float* gamma, const float* beta, const float* mean, const float* var,
                           const float* bias, int C, float eps, float* scale, float* shift, dcb_stream_t stream) {
  DCB_CHECK_ARG(gamma && beta && mean && var && scale && shift && C > 0, "dcb_bn_fold: bad arguments");
  bn_fold_kernel<<<cdiv(C, 128), 128, 0, (cudaStream_t)stream>>>(gamma, beta, mean, var, bias, C, eps, scale, shift);
  g_launches += 1;
  DCB_LAUNCH_OK("bn_fold_kernel");
  return DCB_OK;
}

static int check_c(int C, const char* who) {
  const int vec = (C % 8 == 0 && 256 % (C / 8) == 0) ? 8 : 4;
  if (C < 4 || C % 4 != 0 || C > 2048 || 256 % (C / vec) != 0)
    return fail(DCB_ERR_INVALID_ARGUMENT, "%s: channel count %d unsupported (need C/4 or C/8 to divide 256)", who, C);
  return DCB_OK;
}

// Grid for the two per-channel reductions: a CTA covers rows_par = 256/(C/VEC) rows per pass and should get at
// least one 4-deep unrolled pass (4*rows_par rows); at most 4 CTAs per SM (each CTA ends with 2*C fp64 atomics).
static int bn_reduce_grid(long long M, int C) {
  const int vec = (C % 8 == 0 && 256 % (C / 8) == 0) ? 8 : 4;
  const int rows_par = 256 / (C / vec) > 0 ? 256 / (C / vec) : 1;
  long long grid = (M + 4LL * rows_par - 1) / (4LL * rows_par);
  const int per_sm = policy(DCB_POLICY_BN_CTAS_PER_SM) > 0 ? policy(DCB_POLICY_BN_CTAS_PER_SM) : 4;
  if (grid > (long long)sm_count() * per_sm) grid = (long long)sm_count() * per_sm;
  return grid < 1 ? 1 : (int)grid;
}

extern "C" int dcb_bn_stats(int dtype, const void* x, long long M, int C, double* sums, dcb_stream_t stream) {
  DCB_CHECK_ARG(x && sums && M > 0, "dcb_bn_stats: bad arguments");
  if (int e = check_c(C, "dcb_bn_stats")) return e;
  const int grid = bn_reduce_grid(M, C);
  if (C % 8 == 0 && 256 % (C / 8) == 0) {
    DISPATCH_T(dtype, bn_stats_kernel<T, 8><<<grid, 256, 0, (cudaStream_t)stream>>>((const T*)x, M, C, sums);)
  } else {
    DISPATCH_T(dtype, bn_stats_kernel<T, 4><<<grid, 256, 0, (cudaStream_t)stream>>>((const T*)x, M, C, sums);)
  }
  g_launches += 1;
  DCB_LAUNCH_OK("bn_stats_kernel");
  return DCB_OK;
}

extern "C" int dcb_bn_finalize(const double* sums, long long M, int C, const float* gamma, const float* beta, float eps,
                               float momentum, float* moving_mean, float* moving_var, float* scale, float* shift,
                               float* mean, float* rstd, dcb_stream_t stream) {
  DCB_CHECK_ARG(sums && gamma && beta && scale && shift && mean && rstd && M > 0 && C > 0, "dcb_bn_finalize: bad arguments");
  bn_finalize_kernel<<<cdiv(C, 128), 128, 0, (cudaStream_t)stream>>>(sums, M, C, gamma, beta, eps, momentum, moving_mean,
                                                                     moving_var, scale, shift, mean, rstd);
  g_launches += 1;
  DCB_LAUNCH_OK("bn_finalize_kernel");
  return DCB_OK;
}

extern "C" int dcb_bn_apply(int dtype, const void* x, long long M, int C, const float* scale, const float* shift, int relu,
                            float p_drop, unsigned long long seed, const unsigned long long* seed_dev, unsigned layer, void* y,
                            dcb_stream_t stream) {
  DCB_CHECK_ARG(x && y && scale && shift && M > 0 && C % 4 == 0, "dcb_bn_apply: bad arguments");
  DCB_CHECK_ARG(p_drop >= 0.f && p_drop < 1.f, "dcb_bn_apply: p_drop must be in [0,1)");
  const size_t coef_smem = 2 * (size_t)C * sizeof(float);
  if (C % 8 == 0) {
    DISPATCH_T(dtype, bn_apply_kernel<T, 8><<<ew_grid(M * C / 8, 256), 256, coef_smem, (cudaStream_t)stream>>>(
        (const T*)x, M, C, scale, shift, relu, p_drop, seed, seed_dev, layer, (T*)y);)
  } else {
    DISPATCH_T(dtype, bn_apply_kernel<T, 4><<<ew_grid(M * C / 4, 256), 256, coef_smem, (cudaStream_t)stream>>>(
        (const T*)x, M, C, scale, shift, relu, p_drop, seed, seed_dev, layer, (T*)y);)
  }
  g_launches += 1;
  DCB_LAUNCH_OK("bn_apply_kernel");
  note_kernel(C % 8 == 0 ? "bn_apply_v8" : "bn_apply_v4");
  return DCB_OK;
}

extern "C" int dcb_bn_finalize_apply(int dtype, const void* x, long long M, int C, const double* sums, long long M_total,
                                     const float* gamma, const float* beta, float eps, float momentum, float* moving_mean,
                                     float* moving_var, float* scale, float* shift, float* mean, float* rstd, int relu,
                                     float p_drop, unsigned long long seed, const unsigned long long* seed_dev, unsigned layer,
                                     void* y, dcb_stream_t stream) {
  DCB_CHECK_ARG(x && y && sums && gamma && beta && scale && shift && mean && rstd && M > 0 && C > 0 && C % 4 == 0 && C <= 2048,
                "dcb_bn_finalize_apply: bad arguments (C %d)", C);
  DCB_CHECK_ARG(p_drop >= 0.f && p_drop < 1.f, "dcb_bn_finalize_apply: p_drop %f outside [0, 1)", p_drop);
  if (M_total <= 0) M_total = M;
  const size_t coef_smem = 2 * (size_t)C * sizeof(float);
  if (C % 8 == 0) {
    DISPATCH_T(dtype, bn_finalize_apply_kernel<T, 8><<<ew_grid(M * C / 8, 256), 256, coef_smem, (cudaStream_t)stream>>>(
        (const T*)x, M, C, sums, M_total, gamma, beta, eps, momentum, moving_mean, moving_var, scale, shift, mean, rstd, relu,
        p_drop, seed, seed_dev, layer, (T*)y);)
  } else {
    DISPATCH_T(dtype, bn_finalize_apply_kernel<T, 4><<<ew_grid(M * C / 4, 256), 256, coef_smem, (cudaStream_t)stream>>>(
        (const T*)x, M, C, sums, M_total, gamma, beta, eps, momentum, moving_mean, moving_var, scale, shift, mean, rstd, relu,
        p_drop, seed, seed_dev, layer, (T*)y);)
  }
  g_launches += 1;
  DCB_LAUNCH_OK("bn_finalize_apply_kernel");
  note_kernel(C % 8 == 0 ? "bn_finalize_apply_v8" : "bn_finalize_apply_v4");
  return DCB_OK;
}

extern "C" int dcb_bn_bwd_reduce(int dtype, const float* dy, int ldy, int offy, const void* x, long long M, int C,
                                 const float* scale, const float* shift, const float* mean, const float* rstd,
                                 float p_drop, unsigned long long seed, const unsigned long long* seed_dev, unsigned layer,
                                 double* sums, dcb_stream_t stream) {
  DCB_CHECK_ARG(dy && x && scale && shift && mean && rstd && sums && M > 0, "dcb_bn_bwd_reduce: bad arguments");
  DCB_CHECK_ARG(ldy % 4 == 0 && offy % 4 == 0 && offy + C <= ldy, "dcb_bn_bwd_reduce: bad dy view (ld %d off %d C %d)", ldy, offy, C);
  DCB_CHECK_ARG((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(dy) & 15) == 0, "dcb_bn_bwd_reduce: pointers must be 16-byte aligned");
  if (int e = check_c(C, "dcb_bn_bwd_reduce")) return e;
  const int grid = bn_reduce_grid(M, C);
  if (C % 8 == 0 && 256 % (C / 8) == 0) {
    DISPATCH_T(dtype, bn_bwd_reduce_kernel<T, 8><<<grid, 256, 0, (cudaStream_t)stream>>>(
        (const float*)dy, ldy, offy, (const T*)x, M, C, scale, shift, mean, rstd, p_drop, seed, seed_dev, layer, sums);)
  } else {
    DISPATCH_T(dtype, bn_bwd_reduce_kernel<T, 4><<<grid, 256, 0, (cudaStream_t)stream>>>(
        (const float*)dy, ldy, offy, (const T*)x, M, C, scale, shift, mean, rstd, p_drop, seed, seed_dev, layer, sums);)
  }
  g_launches += 1;
  DCB_LAUNCH_OK("bn_bwd_reduce_kernel");
  note_kernel(C % 8 == 0 && 256 % (C / 8) == 0 ? "bn_bwd_reduce_v8" : "bn_bwd_reduce_v4");
  return DCB_OK;
}

extern "C" int dcb_bn_bwd_apply(int dtype, const float* dy, int ldy, int offy, const void* x, long long M, int C,
                                const float* scale, const float* shift, const float* mean, const float* rstd,
                                float p_drop, unsigned long long seed, const unsigned long long* seed_dev, unsigned layer,
                                const double* sums, long long M_total, float dgb_scale, void* draw, float* dgamma,
                                float* dbeta, dcb_stream_t stream) {
  if (M_total <= 0) M_total = M;
  DCB_CHECK_ARG(dy && x && scale && shift && mean && rstd && sums && draw && M > 0, "dcb_bn_bwd_apply: bad arguments");
  DCB_CHECK_ARG(ldy % 4 == 0 && offy % 4 == 0 && offy + C <= ldy && C % 4 == 0, "dcb_bn_bwd_apply: bad dy view");
  const size_t coef_smem = 5 * (size_t)C * sizeof(float);
  if (C % 8 == 0) {
    DISPATCH_T(dtype, bn_bwd_apply_kernel<T, 8><<<ew_grid(M * C / 8, 256), 256, coef_smem, (cudaStream_t)stream>>>(
        (const float*)dy, ldy, offy, (const T*)x, M, C, scale, shift, mean, rstd, p_drop, seed, seed_dev, layer, sums, M_total, dgb_scale, (T*)draw, dgamma, dbeta);)
  } else {
    DISPATCH_T(dtype, bn_bwd_apply_kernel<T, 4><<<ew_grid(M * C / 4, 256), 256, coef_smem, (cudaStream_t)stream>>>(
        (const float*)dy, ldy, offy, (const T*)x, M, C, scale, shift, mean, rstd, p_drop, seed, seed_dev, layer, sums, M_total, dgb_scale, (T*)draw, dgamma, dbeta);)
  }
  g_launches += 1;
  DCB_LAUNCH_OK("bn_bwd_apply_kernel");
  note_kernel(C % 8 == 0 ? "bn_bwd_apply_v8" : "bn_bwd_apply_v4");
  return DCB_OK;
}

extern "C" int dcb_crop_batch(const long long* img_ptrs, const long long* mask_ptrs, const int* widths, const int* desc,
                              int B, int window, float* x_out, unsigned char* y_out, dcb_stream_t stream) {
  DCB_CHECK_ARG(img_ptrs && mask_ptrs && widths && desc && x_out && y_out && B > 0 && window > 0, "dcb_crop_batch: bad arguments");
  const long long total = (long long)B * window * window;
  crop_batch_kernel<<<ew_grid(total, 256), 256, 0, (cudaStream_t)stream>>>(img_ptrs, mask_ptrs, widths, desc, B, window, x_out,
                                                                           y_out);
  g_launches += 1;
  DCB_LAUNCH_OK("crop_batch_kernel");
  return DCB_OK;
}

extern "C" int dcb_upsample2x(int dtype, const void* x, int N, int h, int w, int C, float p_drop, unsigned long long seed,
                              const unsigned long long* seed_dev, unsigned layer, void* y, dcb_stream_t stream) {
  DCB_CHECK_ARG(x && y && N > 0 && h > 0 && w > 0 && C > 0 && C % 4 == 0, "dcb_upsample2x: bad arguments (C %d)", C);
  DCB_CHECK_ARG(p_drop >= 0.f && p_drop < 1.f, "dcb_upsample2x: p_drop %f outside [0, 1)", p_drop);
  const long long n4 = (long long)N * 4 * h * w * (C / 4);
  DISPATCH_T(dtype, upsample2x_kernel<T><<<ew_grid(n4, 256), 256, 0, (cudaStream_t)stream>>>(
      (const T*)x, N, h, w, C, p_drop, seed, seed_dev, layer, (T*)y);)
  g_launches += 1;
  DCB_LAUNCH_OK("upsample2x_kernel");
  return DCB_OK;
}

extern "C" int dcb_upsample2x_bwd(const float* dy, int ldy, int offy, int N, int h, int w, int C, float p_drop,
                                  unsigned long long seed, const unsigned long long* seed_dev, unsigned layer, float* dx,
                                  dcb_stream_t stream) {
  DCB_CHECK_ARG(dy && dx && N > 0 && h > 0 && w > 0 && C > 0 && C % 4 == 0 && ldy % 4 == 0 && offy % 4 == 0 && offy + C <= ldy,
                "dcb_upsample2x_bwd: bad arguments (C %d ld %d off %d)", C, ldy, offy);
  const long long n4 = (long long)N * h * w * (C / 4);
  upsample2x_bwd_kernel<<<ew_grid(n4, 256), 256, 0, (cudaStream_t)stream>>>(dy, ldy, offy, N, h, w, C, p_drop, seed, seed_dev,
                                                                            layer, dx);
  g_launches += 1;
  DCB_LAUNCH_OK("upsample2x_bwd_kernel");
  return DCB_OK;
}

extern "C" int dcb_maxpool2x2(int dtype, const void* x, int N, int H, int W, int C, void* y, dcb_stream_t stream) {
  DCB_CHECK_ARG(x && y && N > 0 && H > 0 && W > 0 && H % 2 == 0 && W % 2 == 0 && C % 4 == 0, "dcb_maxpool2x2: bad arguments");
  if (C % 8 == 0) {
    DISPATCH_T(dtype, maxpool2x2_v8_kernel<T><<<ew_grid((long long)N * (H / 2) * (W / 2) * (C / 8), 256), 256, 0, (cudaStream_t)stream>>>(
        (const T*)x, N, H, W, C, (T*)y);)
  } else {
    DISPATCH_T(dtype, maxpool2x2_kernel<T><<<ew_grid((long long)N * (H / 2) * (W / 2) * (C / 4), 256), 256, 0, (cudaStream_t)stream>>>(
        (const T*)x, N, H, W, C, (T*)y);)
  }
  g_launches += 1;
  DCB_LAUNCH_OK("maxpool2x2_kernel");
  return DCB_OK;
}

extern "C" int dcb_pool_bwd_add(int dtype, const float* skipgrad, int lds, int offs, const void* y, const void* pooled,
                                const float* dpool, int N, int H, int W, int C, float* out, dcb_stream_t stream) {
  DCB_CHECK_ARG(y && pooled && dpool && out && N > 0 && H % 2 == 0 && W % 2 == 0 && C % 4 == 0, "dcb_pool_bwd_add: bad arguments");
  DCB_CHECK_ARG(!skipgrad || (lds % 4 == 0 && offs % 4 == 0 && offs + C <= lds), "dcb_pool_bwd_add: bad skip-gradient view");
  DISPATCH_T(dtype, {
    return launch(pool_bwd_add_kernel<T>, "pool_bwd_add_kernel", ew_grid((long long)N * (H / 2) * (W / 2) * (C / 4), 256), 256, 0, 0,
                  (cudaStream_t)stream, policy(DCB_POLICY_PDL) != 0, 0, (const float*)skipgrad, lds, offs, (const T*)y,
                  (const T*)pooled, (const float*)dpool, N, H, W, C, (float*)out);
  })
}

extern "C" int dcb_head_fwd(int dtype, const void* x, long long M, int C, const float* w, const float* b, float* logit,
                            float* prob, dcb_stream_t stream) {
  DCB_CHECK_ARG(x && w && b && (logit || prob) && M > 0 && C % 4 == 0 && C <= 512, "dcb_head_fwd: bad arguments");
  DISPATCH_T(dtype, head_fwd_kernel<T><<<ew_grid(M, 256), 256, 0, (cudaStream_t)stream>>>((const T*)x, M, C, w, b, logit, prob);)
  g_launches += 1;
  DCB_LAUNCH_OK("head_fwd_kernel");
  return DCB_OK;
}

extern "C" int dcb_head_loss_fwd(int dtype, const void* x, long long M, int C, const float* w, const float* b,
                                 const uint8_t* yt, float* prob, double* sums, dcb_stream_t stream) {
  DCB_CHECK_ARG(x && w && b && yt && prob && sums && M > 0 && C % 4 == 0 && C <= 512, "dcb_head_loss_fwd: bad arguments");
  DISPATCH_T(dtype, head_loss_fwd_kernel<T><<<ew_grid(M, 256), 256, 0, (cudaStream_t)stream>>>((const T*)x, M, C, w, b, yt, prob, sums);)
  g_launches += 1;
  DCB_LAUNCH_OK("head_loss_fwd_kernel");
  return DCB_OK;
}

extern "C" int dcb_head_loss_bwd(int dtype, const void* x, long long M, int C, const float* w, const uint8_t* yt,
                                 const float* prob, const double* sums, int loss, long long M_total, float* dx,
                                 double* dwb_accum, float* dw_out, float* metrics_out, dcb_stream_t stream) {
  if (M_total <= 0) M_total = M;
  DCB_CHECK_ARG(x && w && yt && prob && sums && dx && dwb_accum && dw_out && metrics_out && M > 0 && C % 4 == 0 && C <= 512,
                "dcb_head_loss_bwd: bad arguments");
  DCB_CHECK_ARG(loss >= 0 && loss <= 3, "dcb_head_loss_bwd: unknown loss id %d", loss);
  int grid = ew_grid(M, 256); if (grid > sm_count() * 4) grid = sm_count() * 4;
  if (C == 32 && (reinterpret_cast<uintptr_t>(x) & 15) == 0) {
    DISPATCH_T(dtype, head_loss_bwd_c32_kernel<T><<<grid, 256, 0, (cudaStream_t)stream>>>((const T*)x, M, w, yt, prob, sums, loss, M_total, (float*)dx, dwb_accum, nullptr, nullptr);)
  } else {
    DISPATCH_T(dtype, head_loss_bwd_kernel<T><<<grid, 256, 0, (cudaStream_t)stream>>>((const T*)x, M, C, w, yt, prob, sums, loss, M_total, (float*)dx, dwb_accum);)
  }
  DCB_LAUNCH_OK("head_loss_bwd_kernel");
  head_metrics_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(sums, M_total, loss, metrics_out, dwb_accum, C, dw_out);
  g_launches += 2;
  DCB_LAUNCH_OK("head_metrics_kernel");
  return DCB_OK;
}

extern "C" int dcb_head_loss_bwd_rank1(int dtype, const void* x, long long M, int C, const float* w, const uint8_t* yt,
                                       const float* prob, const double* sums, int loss, long long M_total, float* gpix,
                                       float* wd_out, double* dwb_accum, float* dw_out, float* metrics_out, dcb_stream_t stream) {
  if (M_total <= 0) M_total = M;
  DCB_CHECK_ARG(x && w && yt && prob && sums && gpix && wd_out && dwb_accum && dw_out && metrics_out && M > 0,
                "dcb_head_loss_bwd_rank1: bad arguments");
  DCB_CHECK_ARG(loss >= 0 && loss <= 3, "dcb_head_loss_bwd_rank1: unknown loss id %d", loss);
  if (C != 32 || (reinterpret_cast<uintptr_t>(x) & 15) != 0)
    return fail(DCB_ERR_UNSUPPORTED, "dcb_head_loss_bwd_rank1: 32 input channels only (got %d); use dcb_head_loss_bwd", C);
  int grid = ew_grid(M, 256); if (grid > sm_count() * 4) grid = sm_count() * 4;
  DISPATCH_T(dtype, head_loss_bwd_c32_kernel<T><<<grid, 256, 0, (cudaStream_t)stream>>>((const T*)x, M, w, yt, prob, sums, loss, M_total, nullptr, dwb_accum, gpix, wd_out);)
  DCB_LAUNCH_OK("head_loss_bwd_kernel");
  head_metrics_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(sums, M_total, loss, metrics_out, dwb_accum, C, dw_out);
  g_launches += 2;
  DCB_LAUNCH_OK("head_metrics_kernel");
  return DCB_OK;
}

static int launch_make_batch(int dtype, const float* s, int hs, int ws, int S, const int* oy, const int* ox, int n_tx,
                             int tile_first, int n_tiles, int first, int count, void* out, dcb_stream_t stream) {
  const bool pdl = policy(DCB_POLICY_PDL) != 0;
  DISPATCH_T(dtype, {
    return launch(tile_make_batch_kernel<T>, "tile_make_batch_kernel", ew_grid((long long)n_tiles * count * S * S, 256), 256, 0, 0,
                  (cudaStream_t)stream, pdl, 0, s, hs, ws, S, oy, ox, n_tx, tile_first, n_tiles, first, count, (T*)out);
  })
}

static int launch_combine(const float* probs, int S, int hs, int ws, const int* oy, const int* ox, const int* cy,
                          const int* cx, int n_ty, int n_tx, int tile_first, int n_tiles, float threshold, int n_aug,
                          double* act, uint8_t* mask, dcb_stream_t stream) {
  return launch(tile_combine_kernel, "tile_combine_kernel", ew_grid((long long)n_tiles * S * S, 256), 256, 0, 0, (cudaStream_t)stream,
                policy(DCB_POLICY_PDL) != 0, 0, probs, S, hs, ws, oy, ox, cy, cx, n_ty, n_tx, tile_first, n_tiles, threshold,
                n_aug, act, mask);
}

extern "C" int dcb_tta_make_batch(int dtype, const float* s, int hs, int ws, int S, int first, int count, void* out,
                                  dcb_stream_t stream) {
  DCB_CHECK_ARG(s && out && hs > 0 && ws > 0 && hs <= S && ws <= S, "dcb_tta_make_batch: image %dx%d does not fit window %d", hs, ws, S);
  DCB_CHECK_ARG(first >= 0 && count > 0 && first + count <= 8, "dcb_tta_make_batch: transforms [%d,%d) out of range", first, first + count);
  return launch_make_batch(dtype, s, hs, ws, S, nullptr, nullptr, 1, 0, 1, first, count, out, stream);
}

extern "C" int dcb_tta_combine(const float* probs, int S, int hs, int ws, float threshold, int n_aug, double* act,
                               uint8_t* mask, dcb_stream_t stream) {
  DCB_CHECK_ARG(probs && mask && hs > 0 && ws > 0 && hs <= S && ws <= S, "dcb_tta_combine: bad arguments");
  DCB_CHECK_ARG(n_aug == 1 || n_aug == 8, "dcb_tta_combine: n_aug must be 1 or 8 (got %d)", n_aug);
  return launch_combine(probs, S, hs, ws, nullptr, nullptr, nullptr, nullptr, 1, 1, 0, 1, threshold, n_aug, act, mask, stream);
}

extern "C" int dcb_tile_make_batch(int dtype, const float* s, int hs, int ws, int T, const int* origins_y,
                                   const int* origins_x, int n_ty, int n_tx, int tile_first, int n_tiles, int first, int count,
                                   void* out, dcb_stream_t stream) {
  DCB_CHECK_ARG(s && out && origins_y && origins_x && hs > 0 && ws > 0 && T > 0 && n_ty > 0 && n_tx > 0,
                "dcb_tile_make_batch: bad arguments");
  DCB_CHECK_ARG(tile_first >= 0 && n_tiles > 0 && (long long)tile_first + n_tiles <= (long long)n_ty * n_tx,
                "dcb_tile_make_batch: tiles [%d,%d) outside the %dx%d plan", tile_first, tile_first + n_tiles, n_ty, n_tx);
  DCB_CHECK_ARG(first >= 0 && count > 0 && first + count <= 8, "dcb_tile_make_batch: transforms [%d,%d) out of range", first, first + count);
  return launch_make_batch(dtype, s, hs, ws, T, origins_y, origins_x, n_tx, tile_first, n_tiles, first, count, out, stream);
}

extern "C" int dcb_tile_combine(const float* probs, int T, int hs, int ws, const int* origins_y, const int* origins_x,
                                const int* cuts_y, const int* cuts_x, int n_ty, int n_tx, int tile_first, int n_tiles,
                                float threshold, int n_aug, double* act, uint8_t* mask, dcb_stream_t stream) {
  DCB_CHECK_ARG(probs && mask && origins_y && origins_x && hs > 0 && ws > 0 && T > 0 && n_ty > 0 && n_tx > 0,
                "dcb_tile_combine: bad arguments");
  DCB_CHECK_ARG((cuts_y || n_ty == 1) && (cuts_x || n_tx == 1), "dcb_tile_combine: a plan with several tiles needs its cuts");
  DCB_CHECK_ARG(tile_first >= 0 && n_tiles > 0 && (long long)tile_first + n_tiles <= (long long)n_ty * n_tx,
                "dcb_tile_combine: tiles [%d,%d) outside the %dx%d plan", tile_first, tile_first + n_tiles, n_ty, n_tx);
  DCB_CHECK_ARG(n_aug == 1 || n_aug == 8, "dcb_tile_combine: n_aug must be 1 or 8 (got %d)", n_aug);
  return launch_combine(probs, T, hs, ws, origins_y, origins_x, cuts_y, cuts_x, n_ty, n_tx, tile_first, n_tiles, threshold,
                        n_aug, act, mask, stream);
}

extern "C" int dcb_adam_step(float* p, const float* g, float* m, float* v, long long n, float lr_t,
                             const float* lr_t_dev, float beta1, float beta2, float eps, dcb_stream_t stream) {
  DCB_CHECK_ARG(p && g && m && v && n > 0, "dcb_adam_step: bad arguments");
  adam_kernel<<<ew_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(p, g, m, v, n, lr_t, lr_t_dev, beta1, beta2, eps);
  g_launches += 1;
  DCB_LAUNCH_OK("adam_kernel");
  return DCB_OK;
}

extern "C" int dcb_step_advance(unsigned long long* state, float lr, float beta1, float beta2, float* lr_t_out,
                                dcb_stream_t stream) {
  DCB_CHECK_ARG(state && lr_t_out, "dcb_step_advance: null pointer");
  step_advance_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(state, lr, beta1, beta2, lr_t_out);
  g_launches += 1;
  DCB_LAUNCH_OK("step_advance_kernel");
  return DCB_OK;
}
