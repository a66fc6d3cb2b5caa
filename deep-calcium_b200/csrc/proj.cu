// K1: per-pixel temporal mean/max projection of a [T][H*W] float32 movie, and
// K1b: summary-image standardisation.
//
// Replaces the streaming loop at deepcalcium/datasets/nf.py:115-130 and
// _summarize_series at deepcalcium/models/neurons/unet_2d_summary.py:227-241.
//
// HBM-bound: the movie is read exactly once (T*P*4 bytes), 2*P*4 bytes are
// written.  Layout: a CTA owns a strip of 4*PXT consecutive pixels; its TG
// thread groups interleave over the frames of the CTA's T-slice, each thread
// issuing U independent 16-byte streaming loads (ld.global.nc.L1::no_allocate)
// before it reduces them.  Sums: the U frames are tree-summed in fp32 and then
// accumulated in fp64 (keeps the mean within ~2e-7 relative of the fp64 truth
// without paying one F2F.F64 per element).  Max uses max.NaN (numpy semantics).
#include <cstdlib>
#include "common.cuh"

namespace dcb {

__device__ __forceinline__ float max_nan(float a, float b) {
  float r;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}

template <int PXT, int TG, int U>
__global__ void __launch_bounds__(PXT * TG)
proj_partial_kernel(const float* __restrict__ movie, int T, long long P, int t_splits,
                    double* __restrict__ psum, float* __restrict__ pmax,
                    float* __restrict__ mean_out, float* __restrict__ max_out, int floor0) {
  const int px = threadIdx.x % PXT;
  const int g = threadIdx.x / PXT;
  const long long p0 = ((long long)blockIdx.x * PXT + px) * 4;   // first of my 4 pixels
  const int split = blockIdx.y;
  const int t_begin = (int)(((long long)T * split) / t_splits);
  const int t_end = (int)(((long long)T * (split + 1)) / t_splits);

  double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
  const float NEG_INF = __int_as_float(0xff800000);
  float m0 = NEG_INF, m1 = NEG_INF, m2 = NEG_INF, m3 = NEG_INF;

  if (p0 < P) {
    const float4* base = reinterpret_cast<const float4*>(movie + p0);
    const long long fstride = P / 4;   // float4 per frame
    int t = t_begin + g;
    for (; t + (U - 1) * TG < t_end; t += U * TG) {
      float4 v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) v[u] = ldg_stream_f4(base + (long long)(t + u * TG) * fstride);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        m0 = max_nan(m0, v[u].x); m1 = max_nan(m1, v[u].y);
        m2 = max_nan(m2, v[u].z); m3 = max_nan(m3, v[u].w);
      }
      // fp32 tree sum of the U frames, then one fp64 accumulate per component
#pragma unroll
      for (int w = 1; w < U; w <<= 1) {
#pragma unroll
        for (int u = 0; u + w < U; u += 2 * w) {
          v[u].x += v[u + w].x; v[u].y += v[u + w].y; v[u].z += v[u + w].z; v[u].w += v[u + w].w;
        }
      }
      s0 += (double)v[0].x; s1 += (double)v[0].y; s2 += (double)v[0].z; s3 += (double)v[0].w;
    }
    for (; t < t_end; t += TG) {
      float4 v = ldg_stream_f4(base + (long long)t * fstride);
      m0 = max_nan(m0, v.x); m1 = max_nan(m1, v.y); m2 = max_nan(m2, v.z); m3 = max_nan(m3, v.w);
      s0 += (double)v.x; s1 += (double)v.y; s2 += (double)v.z; s3 += (double)v.w;
    }
  }

  // combine the TG frame groups of this CTA in a fixed order
  __shared__ double sh_sum[(TG > 1) ? (TG - 1) * PXT * 4 : 1];
  __shared__ float sh_max[(TG > 1) ? (TG - 1) * PXT * 4 : 1];
  if (TG > 1) {
    if (g > 0) {
      double* ds = sh_sum + ((g - 1) * PXT + px) * 4;
      float* dm = sh_max + ((g - 1) * PXT + px) * 4;
      ds[0] = s0; ds[1] = s1; ds[2] = s2; ds[3] = s3;
      dm[0] = m0; dm[1] = m1; dm[2] = m2; dm[3] = m3;
    }
    __syncthreads();
    if (g == 0) {
#pragma unroll
      for (int gg = 1; gg < TG; ++gg) {
        const double* ds = sh_sum + ((gg - 1) * PXT + px) * 4;
        const float* dm = sh_max + ((gg - 1) * PXT + px) * 4;
        s0 += ds[0]; s1 += ds[1]; s2 += ds[2]; s3 += ds[3];
        m0 = max_nan(m0, dm[0]); m1 = max_nan(m1, dm[1]); m2 = max_nan(m2, dm[2]); m3 = max_nan(m3, dm[3]);
      }
    }
  }
  if (g != 0 || p0 >= P) return;

  if (t_splits == 1) {
    const double inv = 1.0 / (double)T;
    float4 mo = make_float4((float)(s0 * inv), (float)(s1 * inv), (float)(s2 * inv), (float)(s3 * inv));
    if (floor0) { m0 = max_nan(m0, 0.f); m1 = max_nan(m1, 0.f); m2 = max_nan(m2, 0.f); m3 = max_nan(m3, 0.f); }
    *reinterpret_cast<float4*>(mean_out + p0) = mo;
    *reinterpret_cast<float4*>(max_out + p0) = make_float4(m0, m1, m2, m3);
  } else {
    double* ps = psum + (long long)split * P + p0;
    reinterpret_cast<double2*>(ps)[0] = make_double2(s0, s1);
    reinterpret_cast<double2*>(ps)[1] = make_double2(s2, s3);
    *reinterpret_cast<float4*>(pmax + (long long)split * P + p0) = make_float4(m0, m1, m2, m3);
  }
}

__global__ void proj_finalize_kernel(const double* __restrict__ psum, const float* __restrict__ pmax,
                                     int t_splits, int T, long long P, float* __restrict__ mean_out,
                                     float* __restrict__ max_out, int floor0) {
  long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  double s = 0;
  float m = __int_as_float(0xff800000);
  for (int k = 0; k < t_splits; ++k) {      // fixed order: deterministic
    s += psum[(long long)k * P + p];
    m = max_nan(m, pmax[(long long)k * P + p]);
  }
  if (floor0) m = max_nan(m, 0.f);
  mean_out[p] = (float)(s / (double)T);
  max_out[p] = m;
}

// ---- int16 movies (the reference's TIFF frames are int16, datasets/nf.py:115-130): half the bytes per frame ----
// A thread owns 8 consecutive pixels (one 16-byte load per frame).  Sums are exact: int32 over the U frames of one
// unrolled pass (U * 32767 < 2^31), then int64; max with the packed signed-16 SIMD max.  Same CTA layout (PXT pixel
// lanes x TG frame groups), same [split][P] double / float partial format and finalize kernel as the fp32 path.
__device__ __forceinline__ uint4 ldg_stream_u4(const uint4* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}

template <int PXT, int TG, int U>
__global__ void __launch_bounds__(PXT * TG)
proj_partial_i16_kernel(const short* __restrict__ movie, int T, long long P, int t_splits, double* __restrict__ psum,
                        float* __restrict__ pmax, float* __restrict__ mean_out, float* __restrict__ max_out, int floor0) {
  const int px = threadIdx.x % PXT;
  const int g = threadIdx.x / PXT;
  const long long p0 = ((long long)blockIdx.x * PXT + px) * 8;   // first of my 8 pixels
  const int split = blockIdx.y;
  const int t_begin = (int)(((long long)T * split) / t_splits);
  const int t_end = (int)(((long long)T * (split + 1)) / t_splits);
  long long s[8];
  uint32_t mx[4];                                                // 4 x packed (int16, int16) running max
#pragma unroll
  for (int i = 0; i < 8; ++i) s[i] = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) mx[i] = 0x80008000u;               // (-32768, -32768)
  if (p0 < P) {
    const uint4* base = reinterpret_cast<const uint4*>(movie + p0);
    const long long fstride = P / 8;                             // uint4 per frame
    auto accumulate = [&](const uint4& v, int (&a)[8]) {
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        mx[i] = __vmaxs2(mx[i], w[i]);
        a[2 * i] += (int)(short)(w[i] & 0xffffu);
        a[2 * i + 1] += (int)w[i] >> 16;
      }
    };
    int t = t_begin + g;
    for (; t + (U - 1) * TG < t_end; t += U * TG) {
      uint4 v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) v[u] = ldg_stream_u4(base + (long long)(t + u * TG) * fstride);
      int a[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
      for (int u = 0; u < U; ++u) accumulate(v[u], a);
#pragma unroll
      for (int i = 0; i < 8; ++i) s[i] += a[i];
    }
    for (; t < t_end; t += TG) {
      const uint4 v = ldg_stream_u4(base + (long long)t * fstride);
      int a[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      accumulate(v, a);
#pragma unroll
      for (int i = 0; i < 8; ++i) s[i] += a[i];
    }
  }
  // combine the TG frame groups of this CTA in a fixed order (integer sums: order does not matter, max neither)
  __shared__ long long sh_sum[(TG > 1) ? (TG - 1) * PXT * 8 : 1];
  __shared__ uint32_t sh_max[(TG > 1) ? (TG - 1) * PXT * 4 : 1];
  if (TG > 1) {
    if (g > 0) {
#pragma unroll
      for (int i = 0; i < 8; ++i) sh_sum[((g - 1) * PXT + px) * 8 + i] = s[i];
#pragma unroll
      for (int i = 0; i < 4; ++i) sh_max[((g - 1) * PXT + px) * 4 + i] = mx[i];
    }
    __syncthreads();
    if (g == 0) {
      for (int gg = 1; gg < TG; ++gg) {
#pragma unroll
        for (int i = 0; i < 8; ++i) s[i] += sh_sum[((gg - 1) * PXT + px) * 8 + i];
#pragma unroll
        for (int i = 0; i < 4; ++i) mx[i] = __vmaxs2(mx[i], sh_max[((gg - 1) * PXT + px) * 4 + i]);
      }
    }
  }
  if (g != 0 || p0 >= P) return;
  float m[8];
#pragma unroll
  for (int i = 0; i < 4; ++i) { m[2 * i] = (float)(short)(mx[i] & 0xffffu); m[2 * i + 1] = (float)((int)mx[i] >> 16); }
  if (t_splits == 1) {
    const double inv = 1.0 / (double)T;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      mean_out[p0 + i] = (float)((double)s[i] * inv);
      max_out[p0 + i] = floor0 ? fmaxf(m[i], 0.f) : m[i];
    }
  } else {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      psum[(long long)split * P + p0 + i] = (double)s[i];
      pmax[(long long)split * P + p0 + i] = m[i];
    }
  }
}

__global__ void proj_scalar_i16_kernel(const short* __restrict__ movie, int T, long long P, float* __restrict__ mean_out,
                                       float* __restrict__ max_out, int floor0) {
  long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  long long s = 0;
  int m = -32768;
  for (int t = 0; t < T; ++t) {
    const int v = movie[(long long)t * P + p];
    s += v;
    m = v > m ? v : m;
  }
  if (floor0 && m < 0) m = 0;
  mean_out[p] = (float)((double)s / (double)T);
  max_out[p] = (float)m;
}

// ---- streaming ingest (SURVEY N4): frames arrive in chunks (TIFF decode -> pinned buffer -> device), the running
// per-pixel state lives on the device: exact int64 sums and the int running max, like the reference's loop at
// datasets/nf.py:126-130 but without its float16 read-modify-write.  One thread per pixel pair group; a pixel is owned
// by exactly one thread, so the accumulation needs no atomics.  PCIe / decode bound, not HBM bound.
__global__ void __launch_bounds__(128)
proj_accum_i16_kernel(const short* __restrict__ chunk, int Tc, long long P, long long* __restrict__ sum, int* __restrict__ mx) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  long long s = sum[p];
  int m = mx[p];
  int t = 0;
  for (; t + 8 <= Tc; t += 8) {
    int v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = chunk[(long long)(t + u) * P + p];
#pragma unroll
    for (int u = 0; u < 8; ++u) { s += v[u]; m = v[u] > m ? v[u] : m; }
  }
  for (; t < Tc; ++t) { const int v = chunk[(long long)t * P + p]; s += v; m = v > m ? v : m; }
  sum[p] = s; mx[p] = m;
}

// bias: value that was subtracted from every pixel before accumulation (unsigned 16-bit frames are shifted into the
// int16 range by -32768); it is restored here in exact integer arithmetic
__global__ void proj_accum_finalize_kernel(const long long* __restrict__ sum, const int* __restrict__ mx, int T, long long P,
                                           float* __restrict__ mean_out, float* __restrict__ max_out, int floor0, int bias) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  int m = mx[p] + bias;
  if (floor0 && m < 0) m = 0;
  mean_out[p] = (float)((double)(sum[p] + (long long)T * bias) / (double)T);
  max_out[p] = (float)m;
}

// generic fallback for P % 4 != 0 (never the benchmark shape): one thread per pixel
__global__ void proj_scalar_kernel(const float* __restrict__ movie, int T, long long P,
                                   float* __restrict__ mean_out, float* __restrict__ max_out, int floor0) {
  long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  double s = 0;
  float m = __int_as_float(0xff800000);
  for (int t = 0; t < T; ++t) {
    float v = movie[(long long)t * P + p];
    s += (double)v;
    m = max_nan(m, v);
  }
  if (floor0) m = max_nan(m, 0.f);
  mean_out[p] = (float)(s / (double)T);
  max_out[p] = m;
}

// ---- standardise: one 1024-thread CTA, three passes over an L2-resident image ----
__device__ double block_sum_1024(double v, double* sh) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) sh[warp] = v;
  __syncthreads();
  double r = (threadIdx.x < (blockDim.x >> 5)) ? sh[threadIdx.x] : 0.0;
  if (warp == 0) {
    r = warp_sum(r);
    if (lane == 0) sh[32] = r;
  }
  __syncthreads();
  return sh[32];
}

__global__ void __launch_bounds__(1024)
standardize_kernel(const float* __restrict__ in, long long n, float* __restrict__ out, double* __restrict__ stats) {
  __shared__ double sh[33];
  double acc = 0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) acc += (double)in[i];
  const double mean = block_sum_1024(acc, sh) / (double)n;
  acc = 0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) { double d = (double)in[i] - mean; acc += d * d; }
  const double var = block_sum_1024(acc, sh) / (double)n;
  const double sd = sqrt(var);
  // the reference does the arithmetic in float32 (np.mean/np.std of a float32 array)
  const float mean_f = (float)mean, sd_f = (float)sd;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) out[i] = (in[i] - mean_f) / sd_f;
  if (stats && threadIdx.x == 0) { stats[0] = mean; stats[1] = sd; }
}

struct ProjVariant { int pxt, tg; };
static const ProjVariant kVariants[] = {{256, 1}, {128, 2}, {64, 4}, {32, 8}};
static const int kNumVariants = 4;
static const int kDefaultVariant = 1;
static const int kU = 8;

static int default_splits(int T, long long P, int variant) {
  const ProjVariant v = kVariants[variant];
  long long strips = (P / 4 + v.pxt - 1) / v.pxt;
  long long target = (long long)sm_count() * 4 * 7;          // ~7 waves of 4 resident CTAs per SM
  long long s = (target + strips - 1) / strips;
  long long max_s = T / (v.tg * kU * 2);                     // keep >= 2 unrolled iterations per group
  if (s > max_s) s = max_s;
  if (s < 1) s = 1;
  if (s > 64) s = 64;
  return (int)s;
}


}  // namespace dcb

using namespace dcb;

extern "C" int dcb_proj_workspace_bytes(int T, int H, int W, size_t* bytes) {
  DCB_CHECK_ARG(bytes != nullptr && T > 0 && H > 0 && W > 0, "dcb_proj_workspace_bytes: bad arguments");
  // enough for the largest split count the library will ever choose (64)
  *bytes = (size_t)64 * (size_t)H * (size_t)W * (sizeof(double) + sizeof(float));
  return DCB_OK;
}

template <int PXT, int TG>
static void launch_partial(const float* movie, int T, long long P, int S, double* psum, float* pmax,
                           float* mean, float* mx, int floor0, cudaStream_t st) {
  dim3 grid((unsigned)((P / 4 + PXT - 1) / PXT), (unsigned)S);
  proj_partial_kernel<PXT, TG, kU><<<grid, PXT * TG, 0, st>>>(movie, T, P, S, psum, pmax, mean, mx, floor0);
}

extern "C" int dcb_proj_mean_max_f32_variant(const float* movie, int T, int H, int W, float* mean, float* mx,
                                             int floor0, void* ws, size_t ws_bytes, int variant, int t_splits,
                                             dcb_stream_t stream) {
  DCB_CHECK_ARG(movie && mean && mx, "dcb_proj_mean_max_f32: null pointer");
  DCB_CHECK_ARG(T > 0 && H > 0 && W > 0, "dcb_proj_mean_max_f32: T,H,W must be positive (got %d,%d,%d)", T, H, W);
  cudaStream_t st = (cudaStream_t)stream;
  const long long P = (long long)H * W;
  if (P % 4 != 0 || (reinterpret_cast<uintptr_t>(movie) & 15) || (reinterpret_cast<uintptr_t>(mean) & 15) ||
      (reinterpret_cast<uintptr_t>(mx) & 15)) {
    proj_scalar_kernel<<<cdiv(P, 256), 256, 0, st>>>(movie, T, P, mean, mx, floor0);
    g_launches += 1;
    DCB_LAUNCH_OK("proj_scalar_kernel");
    return DCB_OK;
  }
  if (variant < 0) variant = kDefaultVariant;
  DCB_CHECK_ARG(variant < kNumVariants, "dcb_proj_mean_max_f32: unknown variant %d", variant);
  int S = t_splits > 0 ? t_splits : default_splits(T, P, variant);
  if (S > T) S = T;
  if (S > 64) S = 64;
  double* psum = nullptr;
  float* pmax = nullptr;
  if (S > 1) {
    size_t need = (size_t)S * P * (sizeof(double) + sizeof(float));
    if (ws == nullptr || ws_bytes < need)
      return fail(DCB_ERR_WORKSPACE, "dcb_proj_mean_max_f32: workspace %zu B < required %zu B", ws_bytes, need);
    DCB_CHECK_ARG((reinterpret_cast<uintptr_t>(ws) & 15) == 0, "dcb_proj_mean_max_f32: workspace must be 16-byte aligned");
    psum = reinterpret_cast<double*>(ws);
    pmax = reinterpret_cast<float*>(psum + (size_t)S * P);
  }
  switch (variant) {
    case 0: launch_partial<256, 1>(movie, T, P, S, psum, pmax, mean, mx, floor0, st); break;
    case 1: launch_partial<128, 2>(movie, T, P, S, psum, pmax, mean, mx, floor0, st); break;
    case 2: launch_partial<64, 4>(movie, T, P, S, psum, pmax, mean, mx, floor0, st); break;
    default: launch_partial<32, 8>(movie, T, P, S, psum, pmax, mean, mx, floor0, st); break;
  }
  g_launches += 1;
  DCB_LAUNCH_OK("proj_partial_kernel");
  if (S > 1) {
    proj_finalize_kernel<<<cdiv(P, 256), 256, 0, st>>>(psum, pmax, S, T, P, mean, mx, floor0);
    g_launches += 1;
    DCB_LAUNCH_OK("proj_finalize_kernel");
  }
  return DCB_OK;
}

extern "C" int dcb_proj_mean_max_f32(const float* movie, int T, int H, int W, float* mean, float* mx, int floor0,
                                     void* ws, size_t ws_bytes, dcb_stream_t stream) {
  return dcb_proj_mean_max_f32_variant(movie, T, H, W, mean, mx, floor0, ws, ws_bytes, -1, 0, stream);
}

template <int PXT, int TG>
static void launch_partial_i16(const short* movie, int T, long long P, int S, double* psum, float* pmax, float* mean, float* mx,
                               int floor0, cudaStream_t st) {
  dim3 grid((unsigned)((P / 8 + PXT - 1) / PXT), (unsigned)S);
  proj_partial_i16_kernel<PXT, TG, kU><<<grid, PXT * TG, 0, st>>>(movie, T, P, S, psum, pmax, mean, mx, floor0);
}

extern "C" int dcb_proj_mean_max_i16(const short* movie, int T, int H, int W, float* mean, float* mx, int floor0, void* ws,
                                     size_t ws_bytes, dcb_stream_t stream) {
  DCB_CHECK_ARG(movie && mean && mx, "dcb_proj_mean_max_i16: null pointer");
  DCB_CHECK_ARG(T > 0 && H > 0 && W > 0, "dcb_proj_mean_max_i16: T,H,W must be positive (got %d,%d,%d)", T, H, W);
  cudaStream_t st = (cudaStream_t)stream;
  const long long P = (long long)H * W;
  if (P % 8 != 0 || (reinterpret_cast<uintptr_t>(movie) & 15)) {
    proj_scalar_i16_kernel<<<cdiv(P, 256), 256, 0, st>>>(movie, T, P, mean, mx, floor0);
    g_launches += 1;
    DCB_LAUNCH_OK("proj_scalar_i16_kernel");
    return DCB_OK;
  }
  // 8 pixels per thread: half as many strips as the fp32 layout of the same variant -> twice the T splits
  const int variant = kDefaultVariant;
  const ProjVariant v = kVariants[variant];
  const long long strips = (P / 8 + v.pxt - 1) / v.pxt;
  // ~3.5 waves of 4 resident CTAs per SM: more T-splits cost more partial-sum traffic than they gain in balance
  // (sweep on B200, 3000 x 512 x 512: 4 splits 5837 GB/s, 8 -> 6214, 12 -> 6156, 17 -> 5820; scripts/proj_i16_sweep.py)
  long long S = ((long long)sm_count() * 4 * 7 / 2 + strips / 2) / strips;
  const long long max_s = T / (v.tg * kU * 2);
  if (policy(DCB_POLICY_PROJ_I16_SPLITS) > 0) S = policy(DCB_POLICY_PROJ_I16_SPLITS);
  if (S > max_s) S = max_s;
  if (S < 1) S = 1;
  if (S > 64) S = 64;
  double* psum = nullptr;
  float* pmax = nullptr;
  if (S > 1) {
    const size_t need = (size_t)S * P * (sizeof(double) + sizeof(float));
    if (ws == nullptr || ws_bytes < need)
      return fail(DCB_ERR_WORKSPACE, "dcb_proj_mean_max_i16: workspace %zu B < required %zu B", ws_bytes, need);
    DCB_CHECK_ARG((reinterpret_cast<uintptr_t>(ws) & 15) == 0, "dcb_proj_mean_max_i16: workspace must be 16-byte aligned");
    psum = reinterpret_cast<double*>(ws);
    pmax = reinterpret_cast<float*>(psum + (size_t)S * P);
  }
  launch_partial_i16<128, 2>(movie, T, P, (int)S, psum, pmax, mean, mx, floor0, st);
  g_launches += 1;
  DCB_LAUNCH_OK("proj_partial_i16_kernel");
  if (S > 1) {
    proj_finalize_kernel<<<cdiv(P, 256), 256, 0, st>>>(psum, pmax, (int)S, T, P, mean, mx, floor0);
    g_launches += 1;
    DCB_LAUNCH_OK("proj_finalize_kernel");
  }
  return DCB_OK;
}

extern "C" int dcb_proj_accum_i16(const short* chunk, int Tc, int H, int W, long long* sum, int* mx, dcb_stream_t stream) {
  DCB_CHECK_ARG(chunk && sum && mx && Tc > 0 && H > 0 && W > 0, "dcb_proj_accum_i16: bad arguments");
  const long long P = (long long)H * W;
  proj_accum_i16_kernel<<<cdiv(P, 128), 128, 0, (cudaStream_t)stream>>>(chunk, Tc, P, sum, mx);
  g_launches += 1;
  DCB_LAUNCH_OK("proj_accum_i16_kernel");
  return DCB_OK;
}

extern "C" int dcb_proj_accum_finalize_biased(const long long* sum, const int* mx, int T, int H, int W, int bias, float* mean,
                                              float* max_out, int floor0, dcb_stream_t stream) {
  DCB_CHECK_ARG(sum && mx && mean && max_out && T > 0 && H > 0 && W > 0, "dcb_proj_accum_finalize: bad arguments");
  const long long P = (long long)H * W;
  proj_accum_finalize_kernel<<<cdiv(P, 256), 256, 0, (cudaStream_t)stream>>>(sum, mx, T, P, mean, max_out, floor0, bias);
  g_launches += 1;
  DCB_LAUNCH_OK("proj_accum_finalize_kernel");
  return DCB_OK;
}

extern "C" int dcb_proj_accum_finalize(const long long* sum, const int* mx, int T, int H, int W, float* mean, float* max_out,
                                       int floor0, dcb_stream_t stream) {
  return dcb_proj_accum_finalize_biased(sum, mx, T, H, W, 0, mean, max_out, floor0, stream);
}

extern "C" int dcb_standardize_f32(const float* in, long long n, float* out, double* stats, dcb_stream_t stream) {
  DCB_CHECK_ARG(in && out && n > 0, "dcb_standardize_f32: bad arguments");
  standardize_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(in, n, out, stats);
  g_launches += 1;
  DCB_LAUNCH_OK("standardize_kernel");
  return DCB_OK;
}
