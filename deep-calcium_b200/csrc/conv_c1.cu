// First layer of the U-Net: Conv2D(3x3,'same') on the 1-channel summary image
// (unet_2d_summary.py:169-172).  K = 9 is far too small for the tensor pipe; the layer is
// bound by writing its [N,H,W,Cout] output, so it runs on CUDA cores with the weights in registers.
#include "elementwise.cuh"
#include "stats_epilogue.cuh"

namespace dcb {
void launch_reduce_splits(const float* part, int splits, size_t n, float* out, cudaStream_t st);

// v2 (round 2).  The first version kept the weights in shared memory and was bound by the shared-memory pipe (ncu: l1tex
// 90 %, 73 us for 8 x 512^2 against a 21 us HBM-write floor).  Here every thread keeps ITS weights in registers: a thread
// owns 8 output channels (9 x 8 weights, scale, shift) of one pixel column and walks down TH rows of a [TH x TW] tile
// whose (TH + 2) x (TW + 2) input window sits in shared memory (zero-filled outside the image = the 'same' padding);
// the 3 x 3 input window slides down in registers (3 shared-memory loads per pixel, broadcast to the COUT / 8 threads of
// that pixel).  The COUT / 8 threads of a pixel write 16 bytes each, so a warp stores a contiguous run of the NHWC row.
__device__ __forceinline__ void cp_async_f32_zfill(float* smem_dst, const float* gsrc, bool valid) {
  const unsigned d = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
  const int n = valid ? 4 : 0;                                // src-size 0: nothing is read, the 4 bytes are zero-filled
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(d), "l"(gsrc), "r"(n) : "memory");
}

// STATS (training forward): every thread also sums its 8 channels' stored (rounded) outputs and their squares; per-CTA sums in
// a fixed order, cross-CTA total by fixed-point integer atomics as in stats_epilogue.cuh (stat_sums[0..COUT) = sum,
// [COUT..2 COUT) = sum of squares, 2^-20 units).
template <typename T, int COUT, bool STATS = false>
__global__ void __launch_bounds__(256, 2)
conv3x3_c1_fwd_kernel(const float* __restrict__ x, int N, int H, int W, const float* __restrict__ w,
                      const float* __restrict__ scale, const float* __restrict__ shift, int relu, T* __restrict__ out,
                      long long* stat_sums = nullptr) {
  constexpr int TPP = COUT / 8;                               // threads per pixel (8 channels = one 16-byte store each)
  constexpr int TW = 256 / TPP;                               // pixel columns per tile
  constexpr int TH = 16;                                      // rows per tile
  constexpr int WIN = (TH + 2) * (TW + 2);
  // The input windows are double buffered and filled with cp.async (zero fill = the 'same' padding): the window of
  // tile i + 1 streams in while tile i is computed.  Without it the kernel spent 30 % of its issue slots waiting for
  // the staging loads (ncu source view, profiles/r2_c1_ncu.txt).
  __shared__ float s_in[2][WIN];
  const int cg = threadIdx.x % TPP, col = threadIdx.x / TPP;
  if (threadIdx.x == 0) pdl_trigger();
  float2 wr[9][4];                                            // this thread's 8 channels of the 9 taps, as fp32 pairs
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int q = 0; q < 4; ++q) wr[t][q] = make_float2(w[t * COUT + cg * 8 + 2 * q], w[t * COUT + cg * 8 + 2 * q + 1]);
  float2 sc2[4], sh2[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    sc2[q] = scale ? make_float2(scale[cg * 8 + 2 * q], scale[cg * 8 + 2 * q + 1]) : make_float2(1.f, 1.f);
    sh2[q] = shift ? make_float2(shift[cg * 8 + 2 * q], shift[cg * 8 + 2 * q + 1]) : make_float2(0.f, 0.f);
  }
  const int tiles_w = (W + TW - 1) / TW, tiles_h = (H + TH - 1) / TH;
  const int num_tiles = N * tiles_h * tiles_w;
  pdl_wait();                                                 // weights / scale / shift above are static; x is not
  auto prefetch = [&](int tile, int buf) {
    if (tile < num_tiles) {
      const int tw = tile % tiles_w, th = (tile / tiles_w) % tiles_h, n = tile / (tiles_w * tiles_h);
      const int h0 = th * TH, w0 = tw * TW;
      const float* img = x + (size_t)n * H * W;
      for (int i = threadIdx.x; i < WIN; i += 256) {
        const int r = i / (TW + 2), c = i - r * (TW + 2);
        const int ih = h0 + r - 1, iw = w0 + c - 1;
        const bool ok = ih >= 0 && ih < H && iw >= 0 && iw < W;
        cp_async_f32_zfill(&s_in[buf][i], ok ? img + (size_t)ih * W + iw : img, ok);
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  float st_s[STATS ? 8 : 1], st_q[STATS ? 8 : 1];
#pragma unroll
  for (int i = 0; i < (STATS ? 8 : 1); ++i) { st_s[i] = 0.f; st_q[i] = 0.f; }
  int buf = 0;
  prefetch(blockIdx.x, 0);
  for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, buf ^= 1) {
    prefetch(tile + gridDim.x, buf ^ 1);
    asm volatile("cp.async.wait_group 1;" ::: "memory");
    __syncthreads();
    const int tw = tile % tiles_w, th = (tile / tiles_w) % tiles_h, n = tile / (tiles_w * tiles_h);
    const int h0 = th * TH, w0 = tw * TW;
    if (w0 + col < W) {
      const float* sp = s_in[buf] + col;                      // window columns col .. col + 2
      float a0 = sp[0], a1 = sp[1], a2 = sp[2];               // input row h - 1
      float b0 = sp[TW + 2], b1 = sp[TW + 3], b2 = sp[TW + 4];   // input row h
      T* orow = out + (((size_t)n * H + h0) * W + (w0 + col)) * COUT + cg * 8;
#pragma unroll 4
      for (int r = 0; r < TH; ++r) {
        if (h0 + r >= H) break;
        const float* s2 = sp + (r + 2) * (TW + 2);
        const float c0 = s2[0], c1 = s2[1], c2 = s2[2];       // input row h + 1
        const float v[9] = {a0, a1, a2, b0, b1, b2, c0, c1, c2};
        float2 acc[4] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f), make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
#pragma unroll
        for (int t = 0; t < 9; ++t) {
          const float2 vv = make_float2(v[t], v[t]);
#pragma unroll
          for (int q = 0; q < 4; ++q) acc[q] = ffma2(vv, wr[t][q], acc[q]);
        }
        float o[8];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float2 y2 = ffma2(acc[q], sc2[q], sh2[q]);
          o[2 * q] = relu ? fmaxf(y2.x, 0.f) : y2.x;
          o[2 * q + 1] = relu ? fmaxf(y2.y, 0.f) : y2.y;
        }
        store8<T>(orow + (size_t)r * W * COUT, o);
        if constexpr (STATS) {
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const float rv = to_f32<T>(from_f32<T>(o[k]));
            st_s[k] += rv; st_q[k] = fmaf(rv, rv, st_q[k]);
          }
        }
        a0 = b0; a1 = b1; a2 = b2; b0 = c0; b1 = c1; b2 = c2;
      }
    }
    __syncthreads();                                          // this window may be overwritten by the prefetch after next
  }
  if constexpr (STATS) {
    // the TW pixel columns of the CTA share each channel group: column-major partials in shared memory, COUT * 2 threads
    // add them in column order -> this CTA's row
    __shared__ float s_red[256 * 17];
#pragma unroll
    for (int k = 0; k < 8; ++k) { s_red[threadIdx.x * 17 + k] = st_s[k]; s_red[threadIdx.x * 17 + 8 + k] = st_q[k]; }
    __syncthreads();
    if (threadIdx.x < 2 * COUT) {
      const int comp = threadIdx.x / COUT, c = threadIdx.x % COUT, g = c >> 3, k = c & 7;
      float acc = 0.f;
      for (int cl = 0; cl < TW; ++cl) acc += s_red[(cl * TPP + g) * 17 + comp * 8 + k];
      tc::stats_add_q(stat_sums, comp * COUT + c, acc);
    }
  }
}

// dW[t][co] = sum_pixels x[pixel + tap t] * dy[pixel][co].  A warp takes 4 consecutive pixels per step:
// lane l reads 4 channels ((l & 7) * 4 ..) of pixel (l >> 3) - one contiguous 256-byte (bf16) row of dy per
// warp load - and keeps 9 taps x 4 channels of partial sums.  Per-CTA partials, then a fixed-order reduce.
template <typename T>
__global__ void __launch_bounds__(256)
conv3x3_c1_wgrad_kernel(const float* __restrict__ x, const T* __restrict__ dy, int N, int H, int W, int Cout,
                        float* __restrict__ part) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int psub = lane >> 3, c4 = (lane & 7) * 4;
  const long long M = (long long)N * H * W;
  const long long per_cta = ((M + gridDim.x - 1) / gridDim.x + 3) & ~3LL;
  const long long m0 = (long long)blockIdx.x * per_cta;
  long long m1 = m0 + per_cta; if (m1 > M) m1 = M;
  __shared__ float red[8][9][32];
  for (int cbase = 0; cbase < Cout; cbase += 32) {
    float acc[9][4];
#pragma unroll
    for (int t = 0; t < 9; ++t) { acc[t][0] = acc[t][1] = acc[t][2] = acc[t][3] = 0.f; }
    const bool cvalid = cbase + c4 < Cout;
    for (long long mb = m0 + warp * 4; mb < m1; mb += 32) {
      const long long m = mb + psub;
      if (m < m1 && cvalid) {
        const int wq = (int)(m % W), hq = (int)((m / W) % H);
        const float* img = x + (m - (long long)hq * W - wq);
        const float4 g = load4<T>(dy + m * Cout + cbase + c4);
#pragma unroll
        for (int t = 0; t < 9; ++t) {
          const int ih = hq + t / 3 - 1, iw = wq + t % 3 - 1;
          const float v = (ih >= 0 && ih < H && iw >= 0 && iw < W) ? __ldg(img + (long long)ih * W + iw) : 0.f;
          acc[t][0] = fmaf(v, g.x, acc[t][0]); acc[t][1] = fmaf(v, g.y, acc[t][1]);
          acc[t][2] = fmaf(v, g.z, acc[t][2]); acc[t][3] = fmaf(v, g.w, acc[t][3]);
        }
      }
    }
    // combine the 4 pixel sub-groups of the warp, then the 8 warps
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float v = acc[t][j];
        v += __shfl_xor_sync(0xffffffffu, v, 8);
        v += __shfl_xor_sync(0xffffffffu, v, 16);
        if (psub == 0) red[warp][t][c4 + j] = v;
      }
    __syncthreads();
    for (int i = threadIdx.x; i < 9 * 32; i += blockDim.x) {
      const int t = i / 32, l = i % 32;
      float sacc = 0.f;
      for (int wv = 0; wv < 8; ++wv) sacc += red[wv][t][l];
      if (cbase + l < Cout) part[((size_t)blockIdx.x * 9 + t) * Cout + cbase + l] = sacc;
    }
    __syncthreads();
  }
}

// The same contraction for Cout == 32, one image row at a time: the three input rows around output row h are staged
// in shared memory once (zero borders = the 'same' padding) instead of nine bounds-checked global loads with 64-bit
// index arithmetic per pixel and lane; a thread owns 4 channels of two neighbouring pixels and slides a 3 x 4 input
// window over them (12 shared-memory reads for 72 FMAs).  The old kernel spent 70 us of the 32-crop step on 9 x 32 outputs.
template <typename T>
__global__ void __launch_bounds__(256)
conv3x3_c1_wgrad_rows_kernel(const float* __restrict__ x, const T* __restrict__ dy, int N, int H, int W, float* __restrict__ part) {
  constexpr int COUT = 32, MAXW = 512;
  __shared__ float s_x[2][3][MAXW + 2];
  __shared__ float red[8][9][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c4 = (threadIdx.x & 7) * 4, pp = (threadIdx.x >> 3) * 2;      // channel quad, first pixel of the pair
  float acc[9][4];
#pragma unroll
  for (int t = 0; t < 9; ++t) { acc[t][0] = acc[t][1] = acc[t][2] = acc[t][3] = 0.f; }
  const int rows = N * H;
  int buf = 0;
  auto stage = [&](int row, int b) {
    const int n = row / H, h = row - n * H;
    const float* img = x + (size_t)n * H * W;
    for (int i = threadIdx.x; i < 3 * (W + 2); i += 256) {
      const int r = i / (W + 2), c = i - r * (W + 2);
      const int ih = h + r - 1, iw = c - 1;
      s_x[b][r][c] = (ih >= 0 && ih < H && iw >= 0 && iw < W) ? __ldg(img + (size_t)ih * W + iw) : 0.f;
    }
  };
  if ((int)blockIdx.x < rows) stage(blockIdx.x, 0);
  __syncthreads();
  for (int row = blockIdx.x; row < rows; row += gridDim.x) {
    if (row + (int)gridDim.x < rows) stage(row + gridDim.x, buf ^ 1);     // next row's window while this one is consumed
    const T* drow = dy + (size_t)row * W * COUT;
    for (int w = pp; w < W; w += 64) {
      const float4 g0 = load4<T>(drow + (size_t)w * COUT + c4);
      const float4 g1 = (w + 1 < W) ? load4<T>(drow + (size_t)(w + 1) * COUT + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const float v0 = s_x[buf][r][w], v1 = s_x[buf][r][w + 1], v2 = s_x[buf][r][w + 2], v3 = s_x[buf][r][w + 3 < W + 2 ? w + 3 : w + 2];
        const float va[3] = {v0, v1, v2}, vb[3] = {v1, v2, v3};
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          float* a = acc[r * 3 + d];
          a[0] = fmaf(va[d], g0.x, a[0]); a[1] = fmaf(va[d], g0.y, a[1]); a[2] = fmaf(va[d], g0.z, a[2]); a[3] = fmaf(va[d], g0.w, a[3]);
          a[0] = fmaf(vb[d], g1.x, a[0]); a[1] = fmaf(vb[d], g1.y, a[1]); a[2] = fmaf(vb[d], g1.z, a[2]); a[3] = fmaf(vb[d], g1.w, a[3]);
        }
      }
    }
    __syncthreads();
    buf ^= 1;
  }
  // combine the 4 pixel pairs of the warp (lanes with the same channel quad), then the 8 warps
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float v = acc[t][j];
      v += __shfl_xor_sync(0xffffffffu, v, 8);
      v += __shfl_xor_sync(0xffffffffu, v, 16);
      if ((lane >> 3) == 0) red[warp][t][c4 + j] = v;
    }
  __syncthreads();
  for (int i = threadIdx.x; i < 9 * 32; i += blockDim.x) {
    const int t = i / 32, l = i % 32;
    float sacc = 0.f;
    for (int wv = 0; wv < 8; ++wv) sacc += red[wv][t][l];
    part[((size_t)blockIdx.x * 9 + t) * COUT + l] = sacc;
  }
}

}  // namespace dcb

using namespace dcb;

template <typename T>
static int launch_c1_fwd(const float* x, int N, int H, int W, const float* w, int Cout, const float* scale,
                         const float* shift, int relu, T* out, cudaStream_t st, long long* stat_sums = nullptr,
                         int* stats_done = nullptr) {
  // persistent: two 256-thread CTAs per SM walk the [16 x (2048 / Cout)]-pixel tiles
  auto tiles = [&](int tw) { return (long long)N * cdiv(H, 16) * cdiv(W, tw); };
  auto grid_for = [&](long long t) { const long long cap = 2LL * sm_count(); return (int)(t < cap ? t : cap); };
  const bool pdl = policy(DCB_POLICY_PDL) != 0;
  if (stats_done) *stats_done = 0;
  if (stat_sums && Cout == 32) {
    if (int e = launch(conv3x3_c1_fwd_kernel<T, 32, true>, "conv3x3_c1_fwd_kernel (stats)", grid_for(tiles(64)), 256, 0, 0, st, pdl, 0,
                       x, N, H, W, w, scale, shift, relu, out, stat_sums))
      return e;
    if (stats_done) *stats_done = 1;
    return DCB_OK;
  }
  const char* name = "conv3x3_c1_fwd_kernel";
  switch (Cout) {
    case 8: return launch(conv3x3_c1_fwd_kernel<T, 8>, name, grid_for(tiles(256)), 256, 0, 0, st, pdl, 0, x, N, H, W, w, scale, shift, relu, out, (long long*)nullptr);
    case 16: return launch(conv3x3_c1_fwd_kernel<T, 16>, name, grid_for(tiles(128)), 256, 0, 0, st, pdl, 0, x, N, H, W, w, scale, shift, relu, out, (long long*)nullptr);
    case 32: return launch(conv3x3_c1_fwd_kernel<T, 32>, name, grid_for(tiles(64)), 256, 0, 0, st, pdl, 0, x, N, H, W, w, scale, shift, relu, out, (long long*)nullptr);
    case 64: return launch(conv3x3_c1_fwd_kernel<T, 64>, name, grid_for(tiles(32)), 256, 0, 0, st, pdl, 0, x, N, H, W, w, scale, shift, relu, out, (long long*)nullptr);
    default: return fail(DCB_ERR_UNSUPPORTED, "dcb_conv3x3_c1_fwd: Cout=%d unsupported (8,16,32,64)", Cout);
  }
}

extern "C" int dcb_conv3x3_c1_fwd(int dtype, const float* x, int N, int H, int W, const float* w, int Cout,
                                  const float* scale, const float* shift, int relu, void* out, dcb_stream_t stream) {
  DCB_CHECK_ARG(x && w && out && N > 0 && H > 0 && W > 0, "dcb_conv3x3_c1_fwd: bad arguments");
  if (dtype == DCB_F32) return launch_c1_fwd<float>(x, N, H, W, w, Cout, scale, shift, relu, (float*)out, (cudaStream_t)stream);
  if (dtype == DCB_BF16)
    return launch_c1_fwd<__nv_bfloat16>(x, N, H, W, w, Cout, scale, shift, relu, (__nv_bfloat16*)out, (cudaStream_t)stream);
  if (dtype == DCB_F16)
    return launch_c1_fwd<__half>(x, N, H, W, w, Cout, scale, shift, relu, (__half*)out, (cudaStream_t)stream);
  return fail(DCB_ERR_INVALID_ARGUMENT, "unknown dtype %d", dtype);
}

// the same + batch statistics of the stored output (training forward); *stats_done = 1 when sums were written by the
// kernel, 0 when this configuration has no statistics epilogue (the conv itself always runs)
extern "C" int dcb_conv3x3_c1_fwd_stats(int dtype, const float* x, int N, int H, int W, const float* w, int Cout,
                                        const float* scale, const float* shift, int relu, void* out, long long* sums_q,
                                        int* stats_done, dcb_stream_t stream) {
  DCB_CHECK_ARG(x && w && out && sums_q && stats_done && N > 0 && H > 0 && W > 0, "dcb_conv3x3_c1_fwd_stats: bad arguments");
  if (dtype == DCB_BF16)
    return launch_c1_fwd<__nv_bfloat16>(x, N, H, W, w, Cout, scale, shift, relu, (__nv_bfloat16*)out, (cudaStream_t)stream, sums_q,
                                        stats_done);
  *stats_done = 0;
  return dcb_conv3x3_c1_fwd(dtype, x, N, H, W, w, Cout, scale, shift, relu, out, stream);
}

static int c1_wgrad_ctas() { return sm_count() * 8; }

extern "C" int dcb_conv3x3_c1_wgrad_workspace_bytes(int Cout, size_t* bytes) {
  DCB_CHECK_ARG(bytes && Cout > 0, "dcb_conv3x3_c1_wgrad_workspace_bytes: bad arguments");
  *bytes = (size_t)c1_wgrad_ctas() * 9 * Cout * sizeof(float);
  return DCB_OK;
}

extern "C" int dcb_conv3x3_c1_wgrad(int dtype, const float* x, const void* dy, int N, int H, int W, int Cout, float* dW,
                                    void* ws, size_t ws_bytes, dcb_stream_t stream) {
  DCB_CHECK_ARG(x && dy && dW && N > 0 && H > 0 && W > 0 && Cout > 0, "dcb_conv3x3_c1_wgrad: bad arguments");
  const bool rows_ok = Cout == 32 && W <= 512 && (reinterpret_cast<uintptr_t>(dy) & 15) == 0;
  // row-staged kernel: two CTAs per SM, each walks whole image rows; otherwise pixel ranges over 8 CTAs per SM
  const int grid = rows_ok ? (2 * sm_count() < N * H ? 2 * sm_count() : N * H) : c1_wgrad_ctas();
  const size_t need = (size_t)grid * 9 * Cout * sizeof(float);
  if (!ws || ws_bytes < need) return fail(DCB_ERR_WORKSPACE, "dcb_conv3x3_c1_wgrad: workspace %zu B < %zu B", ws_bytes, need);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == DCB_F32) {
    if (rows_ok) conv3x3_c1_wgrad_rows_kernel<float><<<grid, 256, 0, st>>>(x, (const float*)dy, N, H, W, (float*)ws);
    else conv3x3_c1_wgrad_kernel<float><<<grid, 256, 0, st>>>(x, (const float*)dy, N, H, W, Cout, (float*)ws);
  } else if (dtype == DCB_BF16) {
    if (rows_ok) conv3x3_c1_wgrad_rows_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(x, (const __nv_bfloat16*)dy, N, H, W, (float*)ws);
    else conv3x3_c1_wgrad_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(x, (const __nv_bfloat16*)dy, N, H, W, Cout, (float*)ws);
  } else return fail(DCB_ERR_INVALID_ARGUMENT, "unknown dtype %d", dtype);
  DCB_LAUNCH_OK("conv3x3_c1_wgrad_kernel");
  const size_t n = (size_t)9 * Cout;
  launch_reduce_splits((const float*)ws, grid, n, dW, st);
  g_launches += 2;
  DCB_LAUNCH_OK("reduce_splits_kernel");
  return DCB_OK;
}
