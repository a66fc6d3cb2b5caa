// fp32 "check mode" contractions on CUDA cores (no tensor cores): the reference
// arithmetic of every Conv2D / Conv2DTranspose in unet_2d_summary.py:154-167 and of
// their Keras-autodiff gradients, restated as one generic tap-GEMM (see tapgeom.h).
// This path exists so that the bf16 tcgen05 kernels can be checked on the GPU against
// an fp32 result (north star: "1e-4 in an fp32 check mode"); it is not the fast path.
#include "common.cuh"
#include "tapgeom.h"

namespace dcb {

constexpr int FM = 64, FN = 64, FK = 16;

struct F32FwdParams {
  TapGeom g;
  const float* src0; const float* src1; int C0, C1;
  const float* B;          // [zsub][ntaps][K][Nout]
  int Nout;
  float* out; int OC;      // output tensor channel count (== Nout here)
  const float* scale; const float* shift; int relu;
};

__global__ void __launch_bounds__(256)
tapgemm_f32_fwd_kernel(const F32FwdParams p) {
  __shared__ float As[FK][FM + 4];
  __shared__ float Bs[FK][FN + 4];
  const TapGeom& g = p.g;
  const int K = p.C0 + p.C1;
  const long long M = (long long)g.N * g.GH * g.GW;
  const long long m0 = (long long)blockIdx.x * FM;
  const int n0 = blockIdx.y * FN;
  const int z = blockIdx.z;
  const float* Bz = p.B + (size_t)z * g.ntaps * K * p.Nout;
  const int ody = g.zsub > 1 ? (z >> 1) : g.ody;
  const int odx = g.zsub > 1 ? (z & 1) : g.odx;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;

  // the 4 positions this thread loads for the A tile: pos = ty + i*16, k = tx
  int img[4], gh[4], gw[4];
  bool mvalid[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    long long m = m0 + ty + i * 16;
    mvalid[i] = m < M;
    long long mm = mvalid[i] ? m : 0;
    gw[i] = (int)(mm % g.GW); mm /= g.GW;
    gh[i] = (int)(mm % g.GH); img[i] = (int)(mm / g.GH);
  }
  // Blocked summation (16-term chunk -> tap -> total) instead of one running fp32 sum over up to 9 * 768 terms: the
  // check mode exists to be compared with float64, and the BatchNorm backward downstream cancels most leading digits
  // of these sums, so the accumulation order matters (measured: per-tensor gradient error 3x lower).
  float acc[4][4] = {};
  for (int tap = 0; tap < g.ntaps; ++tap) {
    float tacc[4][4] = {};
    size_t pixi[4];
    bool ok[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int ih = gh[i] * g.sy + g.dy[tap], iw = gw[i] * g.sx + g.dx[tap];
      ok[i] = mvalid[i] && ih >= 0 && ih < g.IH && iw >= 0 && iw < g.IW;
      pixi[i] = ((size_t)img[i] * g.IH + (ok[i] ? ih : 0)) * g.IW + (ok[i] ? iw : 0);
    }
    for (int k0 = 0; k0 < K; k0 += FK) {
      const int k = k0 + tx;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float v = 0.f;
        if (ok[i] && k < K) {
          const size_t pix = pixi[i];
          v = (k < p.C0) ? p.src0[pix * p.C0 + k] : p.src1[pix * p.C1 + (k - p.C0)];
        }
        As[tx][ty + i * 16] = v;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        int idx = tid + i * 256;
        int nn = idx & 63, kk = idx >> 6;
        float v = 0.f;
        if (k0 + kk < K && n0 + nn < p.Nout) v = Bz[((size_t)tap * K + k0 + kk) * p.Nout + n0 + nn];
        Bs[kk][nn] = v;
      }
      __syncthreads();
      float cacc[4][4] = {};
#pragma unroll
      for (int kk = 0; kk < FK; ++kk) {
        float a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) { a[i] = As[kk][ty * 4 + i]; b[i] = Bs[kk][tx * 4 + i]; }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) cacc[i][j] = fmaf(a[i], b[j], cacc[i][j]);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) tacc[i][j] += cacc[i][j];
      __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] += tacc[i][j];
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    long long m = m0 + ty * 4 + i;
    if (m >= M) continue;
    long long mm = m;
    int w = (int)(mm % g.GW); mm /= g.GW;
    int h = (int)(mm % g.GH); int n = (int)(mm / g.GH);
    size_t opix = ((size_t)n * g.OH + (h * g.osy + ody)) * g.OW + (w * g.osx + odx);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int c = n0 + tx * 4 + j;
      if (c >= p.Nout) continue;
      float v = acc[i][j];
      if (p.scale) v *= p.scale[c];
      if (p.shift) v += p.shift[c];
      if (p.relu) v = fmaxf(v, 0.f);
      p.out[opix * p.OC + c] = v;
    }
  }
}

// wgrad: part[split][tap][k][n] = sum_{m in split} A(m,tap,k) * G(m,n)
struct F32WgradParams {
  TapGeom g;
  const float* src0; const float* src1; int C0, C1;   // gathered operand ("A")
  const float* G; int Nout;                            // per-position operand [M][Nout]
  float* part;                                         // [splits][ntaps][K][Nout]
  int splits;
};

__global__ void __launch_bounds__(256)
tapgemm_f32_wgrad_kernel(const F32WgradParams p) {
  __shared__ float As[FK][FM + 4];   // [m][k]
  __shared__ float Gs[FK][FN + 4];   // [m][n]
  const TapGeom& g = p.g;
  const int K = p.C0 + p.C1;
  const int ktiles = (K + FM - 1) / FM;
  const int k0 = (blockIdx.x % ktiles) * FM;
  const int n0 = (blockIdx.x / ktiles) * FN;
  const int tap = blockIdx.y;
  const int split = blockIdx.z;
  const long long M = (long long)g.N * g.GH * g.GW;
  const long long mb = (M * split) / p.splits, me = (M * (split + 1)) / p.splits;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  float acc[4][4] = {}, bacc[4][4] = {};     // blocked summation: 16 positions -> 1024 positions -> total
  int chunk = 0;
  for (long long mc = mb; mc < me; mc += FK) {
    // A tile: 16 positions x 64 k ; thread loads position (tid/16), k = tx + j*16
    {
      long long m = mc + ty;
      bool okm = m < me;
      long long mm = okm ? m : 0;
      int w = (int)(mm % g.GW); mm /= g.GW;
      int h = (int)(mm % g.GH); int n = (int)(mm / g.GH);
      int ih = h * g.sy + g.dy[tap], iw = w * g.sx + g.dx[tap];
      bool ok = okm && ih >= 0 && ih < g.IH && iw >= 0 && iw < g.IW;
      size_t pix = ((size_t)n * g.IH + (ok ? ih : 0)) * g.IW + (ok ? iw : 0);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        int k = k0 + tx + j * 16;
        float v = 0.f;
        if (ok && k < K) v = (k < p.C0) ? p.src0[pix * p.C0 + k] : p.src1[pix * p.C1 + (k - p.C0)];
        As[ty][tx + j * 16] = v;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        int c = n0 + tx + j * 16;
        float v = 0.f;
        if (okm && c < p.Nout) v = p.G[(size_t)m * p.Nout + c];
        Gs[ty][tx + j * 16] = v;
      }
    }
    __syncthreads();
    float cacc[4][4] = {};
#pragma unroll
    for (int mm = 0; mm < FK; ++mm) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[mm][ty * 4 + i]; b[i] = Gs[mm][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) cacc[i][j] = fmaf(a[i], b[j], cacc[i][j]);
    }
    const bool flush = (++chunk & 63) == 0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        bacc[i][j] += cacc[i][j];
        if (flush) { acc[i][j] += bacc[i][j]; bacc[i][j] = 0.f; }
      }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] += bacc[i][j];
  float* dst = p.part + ((size_t)split * g.ntaps + tap) * K * p.Nout;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int k = k0 + ty * 4 + i;
    if (k >= K) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int c = n0 + tx * 4 + j;
      if (c < p.Nout) dst[(size_t)k * p.Nout + c] = acc[i][j];
    }
  }
}

// out[i] = sum_s part[s][i]   (fixed order -> deterministic)
__global__ void reduce_splits_kernel(const float* __restrict__ part, int splits, size_t n, float* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int k = 0; k < splits; ++k) s += part[(size_t)k * n + i];
  out[i] = s;
}

// many splits over a small tensor (the strip wgrad's one-partial-per-CTA layout): E elements x (256 / E) split
// lanes per CTA, lane j sums splits j, j+L, ... and the L lane sums are combined in a fixed order (deterministic)
template <int E>
__global__ void __launch_bounds__(256)
reduce_splits_wide_kernel(const float* __restrict__ part, int splits, size_t n, float* __restrict__ out) {
  constexpr int L = 256 / E;
  __shared__ float s_part[L][E];
  const int e = threadIdx.x % E, j = threadIdx.x / E;
  const size_t i = (size_t)blockIdx.x * E + e;
  float a0 = 0.f, a1 = 0.f;
  if (i < n) {
    int k = j;
    for (; k + L < splits; k += 2 * L) { a0 += part[(size_t)k * n + i]; a1 += part[(size_t)(k + L) * n + i]; }
    if (k < splits) a0 += part[(size_t)k * n + i];
  }
  s_part[j][e] = a0 + a1;
  __syncthreads();
  if (j == 0 && i < n) {
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < L; ++q) s += s_part[q][e];
    out[i] = s;
  }
}

void launch_reduce_splits(const float* part, int splits, size_t n, float* out, cudaStream_t st) {
  // split lanes per element: enough to hide the dependent-load chain, few enough that the grid stays small
  if (splits >= 64 && n < 4096) reduce_splits_wide_kernel<8><<<cdiv((long long)n, 8), 256, 0, st>>>(part, splits, n, out);
  else if (splits >= 32) reduce_splits_wide_kernel<32><<<cdiv((long long)n, 32), 256, 0, st>>>(part, splits, n, out);
  else if (splits >= 8) reduce_splits_wide_kernel<128><<<cdiv((long long)n, 128), 256, 0, st>>>(part, splits, n, out);
  else reduce_splits_kernel<<<cdiv((long long)n, 256), 256, 0, st>>>(part, splits, n, out);
}

// same reduction for a partial tensor of nrows x row_len elements whose rows land out_row_stride apart in `out`
// (a K-block of a larger dW[tap][K_total][N]): fixed-order sum over the splits
__global__ void __launch_bounds__(256)
reduce_splits_rows_kernel(const float* __restrict__ part, int splits, int nrows, size_t row_len, float* __restrict__ out,
                          size_t out_row_stride) {
  constexpr int E = 32, L = 8;
  __shared__ float s_part[L][E];
  const int e = threadIdx.x % E, j = threadIdx.x / E;
  const size_t n = (size_t)nrows * row_len;
  const size_t i = (size_t)blockIdx.x * E + e;
  float a0 = 0.f, a1 = 0.f;
  if (i < n) {
    int k = j;
    for (; k + L < splits; k += 2 * L) { a0 += part[(size_t)k * n + i]; a1 += part[(size_t)(k + L) * n + i]; }
    if (k < splits) a0 += part[(size_t)k * n + i];
  }
  s_part[j][e] = a0 + a1;
  __syncthreads();
  if (j == 0 && i < n) {
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < L; ++q) s += s_part[q][e];
    out[(i / row_len) * out_row_stride + i % row_len] = s;
  }
}

void launch_reduce_splits_rows(const float* part, int splits, int nrows, size_t row_len, float* out, size_t out_row_stride,
                               cudaStream_t st) {
  if (out_row_stride == row_len) { launch_reduce_splits(part, splits, (size_t)nrows * row_len, out, st); return; }
  reduce_splits_rows_kernel<<<cdiv((long long)((size_t)nrows * row_len), 32), 256, 0, st>>>(part, splits, nrows, row_len, out,
                                                                                           out_row_stride);
}

void geom_conv3x3(TapGeom& g, int N, int H, int W) {
  memset(&g, 0, sizeof(g));
  g.N = N; g.IH = H; g.IW = W; g.GH = H; g.GW = W; g.sy = g.sx = 1; g.ntaps = 9;
  for (int t = 0; t < 9; ++t) { g.dy[t] = t / 3 - 1; g.dx[t] = t % 3 - 1; }
  g.OH = H; g.OW = W; g.osy = g.osx = 1; g.zsub = 1;
}
void geom_convT_fwd(TapGeom& g, int N, int h, int w) {     // input h x w -> output 2h x 2w
  memset(&g, 0, sizeof(g));
  g.N = N; g.IH = h; g.IW = w; g.GH = h; g.GW = w; g.sy = g.sx = 1; g.ntaps = 1;
  g.OH = 2 * h; g.OW = 2 * w; g.osy = g.osx = 2; g.zsub = 4;
}
void geom_convT_dgrad(TapGeom& g, int N, int h, int w) {   // gathers dy (2h x 2w) -> dx (h x w)
  memset(&g, 0, sizeof(g));
  g.N = N; g.IH = 2 * h; g.IW = 2 * w; g.GH = h; g.GW = w; g.sy = g.sx = 2; g.ntaps = 4;
  for (int t = 0; t < 4; ++t) { g.dy[t] = t / 2; g.dx[t] = t % 2; }
  g.OH = h; g.OW = w; g.osy = g.osx = 1; g.zsub = 1;
}

int run_f32_fwd(const TapGeom& g, const float* s0, int C0, const float* s1, int C1, const float* B, int Nout,
                float* out, const float* scale, const float* shift, int relu, cudaStream_t st) {
  F32FwdParams p;
  p.g = g; p.src0 = s0; p.src1 = s1; p.C0 = C0; p.C1 = C1; p.B = B; p.Nout = Nout; p.out = out; p.OC = Nout;
  p.scale = scale; p.shift = shift; p.relu = relu;
  long long M = (long long)g.N * g.GH * g.GW;
  dim3 grid((unsigned)cdiv(M, FM), (unsigned)cdiv(Nout, FN), (unsigned)(g.zsub > 1 ? g.zsub : 1));
  tapgemm_f32_fwd_kernel<<<grid, 256, 0, st>>>(p);
  g_launches += 1;
  DCB_LAUNCH_OK("tapgemm_f32_fwd_kernel");
  return DCB_OK;
}

int f32_wgrad_splits(const TapGeom& g, int K, int Nout) {
  long long M = (long long)g.N * g.GH * g.GW;
  long long tiles = (long long)cdiv(K, FM) * cdiv(Nout, FN) * g.ntaps;
  long long s = (sm_count() * 8 + tiles - 1) / tiles;
  long long maxs = M / 64; if (maxs < 1) maxs = 1;
  if (s > maxs) s = maxs;
  if (s > 256) s = 256;
  if (s < 1) s = 1;
  return (int)s;
}

int run_f32_wgrad(const TapGeom& g, const float* s0, int C0, const float* s1, int C1, const float* G, int Nout,
                  float* dW, void* ws, size_t ws_bytes, cudaStream_t st) {
  const int K = C0 + C1;
  const int S = f32_wgrad_splits(g, K, Nout);
  const size_t n = (size_t)g.ntaps * K * Nout;
  if (ws == nullptr || ws_bytes < (size_t)S * n * sizeof(float))
    return fail(DCB_ERR_WORKSPACE, "wgrad (fp32): workspace %zu B < required %zu B", ws_bytes, (size_t)S * n * sizeof(float));
  F32WgradParams p;
  p.g = g; p.src0 = s0; p.src1 = s1; p.C0 = C0; p.C1 = C1; p.G = G; p.Nout = Nout;
  p.part = reinterpret_cast<float*>(ws); p.splits = S;
  dim3 grid((unsigned)(cdiv(K, FM) * cdiv(Nout, FN)), (unsigned)g.ntaps, (unsigned)S);
  tapgemm_f32_wgrad_kernel<<<grid, 256, 0, st>>>(p);
  DCB_LAUNCH_OK("tapgemm_f32_wgrad_kernel");
  launch_reduce_splits(p.part, S, n, dW, st);
  g_launches += 2;
  DCB_LAUNCH_OK("reduce_splits_kernel");
  return DCB_OK;
}

}  // namespace dcb
