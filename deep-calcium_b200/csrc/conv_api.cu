// C-ABI entry points of the dense contractions (conv3x3 / convT2x2, fwd / dgrad / wgrad)
// and the weight-layout preparation.  DCB_F32 routes to the CUDA-core check kernels
// (tapgemm_f32.cu), DCB_BF16 to the tcgen05/TMEM/TMA kernels (tapgemm_tc.cu).
#include "common.cuh"
#include "tapgeom.h"
#include <cuda_fp16.h>

namespace dcb {

void geom_conv3x3(TapGeom& g, int N, int H, int W);
void geom_convT_fwd(TapGeom& g, int N, int h, int w);
void geom_convT_dgrad(TapGeom& g, int N, int h, int w);
int run_f32_fwd(const TapGeom& g, const float* s0, int C0, const float* s1, int C1, const float* B, int Nout,
                float* out, const float* scale, const float* shift, int relu, cudaStream_t st);
int f32_wgrad_splits(const TapGeom& g, int K, int Nout);
int run_f32_wgrad(const TapGeom& g, const float* s0, int C0, const float* s1, int C1, const float* G, int Nout,
                  float* dW, void* ws, size_t ws_bytes, cudaStream_t st);

// tcgen05 path (tapgemm_tc.cu)
struct TcFusion {
  const float* head_kernel; const float* head_bias; float* logit; float* prob; int need_y; void* pool_out;
};
struct TcStats { long long* sums; int done; };
int run_tc_fwd(const TapGeom& g, const void* s0, int C0, const void* s1, int C1, const void* B, int Nout, void* out,
               const float* scale, const float* shift, int relu, int out_f32, cudaStream_t st, const TcFusion* fuse = nullptr,
               TcStats* stats = nullptr);
int run_tc_wgrad(const TapGeom& g, const void* s0, int C0, const void* s1, int C1, const void* G, int Nout, float* dW,
                 void* ws, size_t ws_bytes, cudaStream_t st);
size_t tc_wgrad_workspace(const TapGeom& g, int K, int Nout);

// ---- weight preparation ----
// conv3x3: w[t][ci][co] (t = kh*3+kw)
template <typename T>
__global__ void prep_conv3x3_kernel(const float* __restrict__ w, int Cin, int Cout, T* __restrict__ wf,
                                    T* __restrict__ wd, int nmajor) {
  const long long n = 9LL * Cin * Cout;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int co = (int)(i % Cout), ci = (int)((i / Cout) % Cin), t = (int)(i / ((long long)Cout * Cin));
    const float v = w[i];
    if (nmajor) {
      if (wf) wf[((long long)co * 9 + t) * Cin + ci] = from_f32<T>(v);            // [Cout][9][Cin]
      if (wd) wd[((long long)ci * 9 + (8 - t)) * Cout + co] = from_f32<T>(v);      // [Cin][9][Cout], taps flipped
    } else {
      if (wf) wf[i] = from_f32<T>(v);                                              // [9][Cin][Cout]
      if (wd) wd[((long long)(8 - t) * Cout + co) * Cin + ci] = from_f32<T>(v);    // [9][Cout][Cin], taps flipped
    }
  }
}
// convT: w[t][co][ci] (t = a*2+b)
template <typename T>
__global__ void prep_convT_kernel(const float* __restrict__ w, int Cin, int Cout, T* __restrict__ wf,
                                  T* __restrict__ wd, int nmajor) {
  const long long n = 4LL * Cin * Cout;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int ci = (int)(i % Cin), co = (int)((i / Cin) % Cout), t = (int)(i / ((long long)Cout * Cin));
    const float v = w[i];
    if (nmajor) {
      if (wf) wf[i] = from_f32<T>(v);                                              // [4][Cout][Cin]
      if (wd) wd[((long long)ci * 4 + t) * Cout + co] = from_f32<T>(v);            // [Cin][4][Cout]
    } else {
      if (wf) wf[((long long)t * Cin + ci) * Cout + co] = from_f32<T>(v);          // [4][Cin][Cout]
      if (wd) wd[i] = from_f32<T>(v);                                              // [4][Cout][Cin]
    }
  }
}

// all layers of a model in ONE launch: the per-step refresh of the bf16 kernel-layout copies after the optimizer update is
// ~20 tiny launches otherwise.  desc (device memory, 5 x int64 per layer):
// {w, w_fwd (or 0), w_dgrad (or 0), Cin | Cout << 32, kind (0 conv3x3, 1 convT2x2)}
// Work items = 32 x 32 tiles (or 1024-element runs of a layer that has no such tiles) numbered across ALL layers, walked
// grid-stride: a launch shaped (96 CTAs, layer) gave the 2.4 M-element bottom layers 24 tiles per CTA and left most CTAs
// of the small layers idle (67 us for 62 MB of traffic).
constexpr int PREP_MAX_LAYERS = 64;
template <typename T>
__global__ void __launch_bounds__(256)
prep_batch_kernel(const long long* __restrict__ desc, int count, int nmajor) {
  __shared__ int s_first[PREP_MAX_LAYERS + 1];          // first work item of every layer
  __shared__ float tile[32][33];
  if (threadIdx.x == 0) {
    int acc = 0;
    for (int l = 0; l < count; ++l) {
      const long long* d = desc + 5LL * l;
      const int Cin = (int)(d[3] & 0xffffffffLL), Cout = (int)(d[3] >> 32);
      const bool convT = d[4] != 0;
      const int taps = convT ? 4 : 9, R = convT ? Cout : Cin, C = convT ? Cin : Cout;
      s_first[l] = acc;
      acc += (nmajor && R % 32 == 0 && C % 32 == 0) ? taps * (R / 32) * (C / 32) : (taps * Cin * Cout + 1023) / 1024;
    }
    s_first[count] = acc;
  }
  __syncthreads();
  const int total = s_first[count];
  int l = 0;
  for (int item = blockIdx.x; item < total; item += gridDim.x) {
    while (item >= s_first[l + 1]) ++l;                  // items are visited in ascending order
    const long long* d = desc + 5LL * l;
    const float* w = reinterpret_cast<const float*>(d[0]);
    T* wf = reinterpret_cast<T*>(d[1]);
    T* wd = reinterpret_cast<T*>(d[2]);
    const int Cin = (int)(d[3] & 0xffffffffLL), Cout = (int)(d[3] >> 32);
    const bool convT = d[4] != 0;
    const int taps = convT ? 4 : 9;
    // The source is [tap][R][C] with C contiguous (conv: R = Cin, C = Cout; convT: R = Cout, C = Cin).  One of the two
    // bf16 copies keeps C innermost, the other one has R innermost: 32 x 32 tiles go through shared memory so that both
    // are written with contiguous runs (the naive element-wise version scattered 2-byte stores: 109 us per step).
    const int R = convT ? Cout : Cin, C = convT ? Cin : Cout;
    const int tl = item - s_first[l];
    if (nmajor && R % 32 == 0 && C % 32 == 0) {
      const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;          // 32 x 8
      const int tr = R / 32, tc = C / 32;
      const int t = tl / (tr * tc), r0 = (tl / tc) % tr * 32, c0 = (tl % tc) * 32;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int r = r0 + ty + 8 * q, c = c0 + tx;
        const float v = w[((long long)t * R + r) * C + c];
        tile[ty + 8 * q][tx] = v;
        // C-innermost copy: conv w_dgrad [Cin][9 flipped][Cout], convT w_fwd [4][Cout][Cin]
        if (!convT) { if (wd) wd[((long long)r * 9 + (8 - t)) * C + c] = from_f32<T>(v); }
        else if (wf) wf[((long long)t * R + r) * C + c] = from_f32<T>(v);
      }
      __syncthreads();
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int c = c0 + ty + 8 * q, r = r0 + tx;
        const float v = tile[tx][ty + 8 * q];
        // R-innermost copy: conv w_fwd [Cout][9][Cin], convT w_dgrad [Cin][4][Cout]
        if (!convT) { if (wf) wf[((long long)c * 9 + t) * R + r] = from_f32<T>(v); }
        else if (wd) wd[((long long)c * 4 + t) * R + r] = from_f32<T>(v);
      }
      __syncthreads();
      continue;
    }
    const long long n = (long long)taps * Cin * Cout;
    for (long long i = (long long)tl * 1024 + threadIdx.x; i < n && i < (long long)(tl + 1) * 1024; i += blockDim.x) {
      const float v = w[i];
      if (!convT) {
        const int co = (int)(i % Cout), ci = (int)((i / Cout) % Cin), t = (int)(i / ((long long)Cout * Cin));
        if (nmajor) {
          if (wf) wf[((long long)co * 9 + t) * Cin + ci] = from_f32<T>(v);
          if (wd) wd[((long long)ci * 9 + (8 - t)) * Cout + co] = from_f32<T>(v);
        } else {
          if (wf) wf[i] = from_f32<T>(v);
          if (wd) wd[((long long)(8 - t) * Cout + co) * Cin + ci] = from_f32<T>(v);
        }
      } else {
        const int ci = (int)(i % Cin), co = (int)((i / Cin) % Cout), t = (int)(i / ((long long)Cout * Cin));
        if (nmajor) {
          if (wf) wf[i] = from_f32<T>(v);
          if (wd) wd[((long long)ci * 4 + t) * Cout + co] = from_f32<T>(v);
        } else {
          if (wf) wf[((long long)t * Cin + ci) * Cout + co] = from_f32<T>(v);
          if (wd) wd[i] = from_f32<T>(v);
        }
      }
    }
  }
}

}  // namespace dcb

using namespace dcb;

extern "C" int dcb_prep_weights_batch(int dtype, const long long* desc_dev, int count, dcb_stream_t stream) {
  DCB_CHECK_ARG(desc_dev && count > 0 && count <= PREP_MAX_LAYERS, "dcb_prep_weights_batch: bad arguments (at most %d layers)", PREP_MAX_LAYERS);
  const int grid = 8 * sm_count();
  if (dtype == DCB_F32) prep_batch_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(desc_dev, count, 0);
  else if (dtype == DCB_BF16) prep_batch_kernel<__nv_bfloat16><<<grid, 256, 0, (cudaStream_t)stream>>>(desc_dev, count, 1);
  else if (dtype == DCB_F16) prep_batch_kernel<__half><<<grid, 256, 0, (cudaStream_t)stream>>>(desc_dev, count, 1);
  else return fail(DCB_ERR_INVALID_ARGUMENT, "unknown dtype %d", dtype);
  g_launches += 1;
  DCB_LAUNCH_OK("prep_batch_kernel");
  return DCB_OK;
}

extern "C" int dcb_prep_conv3x3_weights(int dtype, const float* w, int Cin, int Cout, void* w_fwd, void* w_dgrad,
                                        dcb_stream_t stream) {
  DCB_CHECK_ARG(w && Cin > 0 && Cout > 0 && (w_fwd || w_dgrad), "dcb_prep_conv3x3_weights: bad arguments");
  const long long n = 9LL * Cin * Cout;
  const int grid = cdiv(n, 256) > 4096 ? 4096 : cdiv(n, 256);
  if (dtype == DCB_F32)
    prep_conv3x3_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(w, Cin, Cout, (float*)w_fwd, (float*)w_dgrad, 0);
  else if (dtype == DCB_BF16)
    prep_conv3x3_kernel<__nv_bfloat16><<<grid, 256, 0, (cudaStream_t)stream>>>(w, Cin, Cout, (__nv_bfloat16*)w_fwd,
                                                                              (__nv_bfloat16*)w_dgrad, 1);
  else if (dtype == DCB_F16)
    prep_conv3x3_kernel<__half><<<grid, 256, 0, (cudaStream_t)stream>>>(w, Cin, Cout, (__half*)w_fwd, (__half*)w_dgrad, 1);
  else return fail(DCB_ERR_INVALID_ARGUMENT, "unknown dtype %d", dtype);
  g_launches += 1;
  DCB_LAUNCH_OK("prep_conv3x3_kernel");
  return DCB_OK;
}

extern "C" int dcb_prep_convT2x2_weights(int dtype, const float* w, int Cin, int Cout, void* w_fwd, void* w_dgrad,
                                         dcb_stream_t stream) {
  DCB_CHECK_ARG(w && Cin > 0 && Cout > 0 && (w_fwd || w_dgrad), "dcb_prep_convT2x2_weights: bad arguments");
  const long long n = 4LL * Cin * Cout;
  const int grid = cdiv(n, 256) > 4096 ? 4096 : cdiv(n, 256);
  if (dtype == DCB_F32)
    prep_convT_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(w, Cin, Cout, (float*)w_fwd, (float*)w_dgrad, 0);
  else if (dtype == DCB_BF16)
    prep_convT_kernel<__nv_bfloat16><<<grid, 256, 0, (cudaStream_t)stream>>>(w, Cin, Cout, (__nv_bfloat16*)w_fwd,
                                                                            (__nv_bfloat16*)w_dgrad, 1);
  else if (dtype == DCB_F16)
    prep_convT_kernel<__half><<<grid, 256, 0, (cudaStream_t)stream>>>(w, Cin, Cout, (__half*)w_fwd, (__half*)w_dgrad, 1);
  else return fail(DCB_ERR_INVALID_ARGUMENT, "unknown dtype %d", dtype);
  g_launches += 1;
  DCB_LAUNCH_OK("prep_convT_kernel");
  return DCB_OK;
}

extern "C" int dcb_conv3x3_fwd(int dtype, const void* src0, int C0, const void* src1, int C1, int N, int H, int W,
                               const void* wgt, int Cout, const float* scale, const float* shift, int relu, void* out,
                               dcb_stream_t stream) {
  DCB_CHECK_ARG(src0 && wgt && out, "dcb_conv3x3_fwd: null pointer");
  DCB_CHECK_ARG(N > 0 && H > 0 && W > 0 && C0 > 0 && C1 >= 0 && Cout > 0 && (C1 == 0 || src1),
                "dcb_conv3x3_fwd: bad shape N=%d H=%d W=%d C0=%d C1=%d Cout=%d", N, H, W, C0, C1, Cout);
  TapGeom g;
  geom_conv3x3(g, N, H, W);
  g.f16 = (dtype == DCB_F16);
  if (dtype == DCB_F32)
    return run_f32_fwd(g, (const float*)src0, C0, (const float*)src1, C1, (const float*)wgt, Cout, (float*)out, scale,
                       shift, relu, (cudaStream_t)stream);
  if (dtype == DCB_BF16 || dtype == DCB_F16)
    return run_tc_fwd(g, src0, C0, src1, C1, wgt, Cout, out, scale, shift, relu, 0, (cudaStream_t)stream);
  return fail(DCB_ERR_INVALID_ARGUMENT, "unknown dtype %d", dtype);
}

extern "C" int dcb_conv3x3_fwd_fused(int dtype, const void* src0, int C0, const void* src1, int C1, int N, int H, int W,
                                     const void* wgt, int Cout, const float* scale, const float* shift, int relu, void* out,
                                     const dcb_conv_fusion_t* fuse, dcb_stream_t stream) {
  DCB_CHECK_ARG(src0 && wgt && out && fuse, "dcb_conv3x3_fwd_fused: null pointer");
  DCB_CHECK_ARG(N > 0 && H > 0 && W > 0 && C0 > 0 && C1 >= 0 && Cout > 0 && (C1 == 0 || src1), "dcb_conv3x3_fwd_fused: bad shape");
  DCB_CHECK_ARG(!fuse->head_kernel || (fuse->head_bias && (fuse->logit || fuse->prob)), "dcb_conv3x3_fwd_fused: incomplete head arguments");
  DCB_CHECK_ARG(!fuse->pool_out || (H % 2 == 0 && W % 2 == 0), "dcb_conv3x3_fwd_fused: pooling needs even H and W");
  if (dtype == DCB_BF16 || dtype == DCB_F16) {
    TapGeom g;
    geom_conv3x3(g, N, H, W);
  g.f16 = (dtype == DCB_F16);
    TcFusion f = {fuse->head_kernel, fuse->head_bias, fuse->logit, fuse->prob, fuse->need_y, fuse->pool_out};
    const int rc = run_tc_fwd(g, src0, C0, src1, C1, wgt, Cout, out, scale, shift, relu, 0, (cudaStream_t)stream, &f);
    if (rc != DCB_ERR_UNSUPPORTED) return rc;
  }
  // unfused composition (fp32 check mode, or a shape the fused epilogue does not cover)
  if (int e = dcb_conv3x3_fwd(dtype, src0, C0, src1, C1, N, H, W, wgt, Cout, scale, shift, relu, out, stream)) return e;
  if (fuse->pool_out)
    if (int e = dcb_maxpool2x2(dtype, out, N, H, W, Cout, fuse->pool_out, stream)) return e;
  if (fuse->head_kernel)
    if (int e = dcb_head_fwd(dtype, out, (long long)N * H * W, Cout, fuse->head_kernel, fuse->head_bias, fuse->logit, fuse->prob, stream)) return e;
  return DCB_OK;
}

extern "C" int dcb_conv3x3_fwd_stats(int dtype, const void* src0, int C0, const void* src1, int C1, int N, int H, int W,
                                     const void* wgt, int Cout, const float* scale, const float* shift, int relu, void* out,
                                     long long* sums_q, int* stats_done, dcb_stream_t stream) {
  DCB_CHECK_ARG(src0 && wgt && out && sums_q && stats_done, "dcb_conv3x3_fwd_stats: null pointer");
  DCB_CHECK_ARG(N > 0 && H > 0 && W > 0 && C0 > 0 && C1 >= 0 && Cout > 0 && (C1 == 0 || src1), "dcb_conv3x3_fwd_stats: bad shape");
  *stats_done = 0;
  if (dtype != DCB_BF16) return dcb_conv3x3_fwd(dtype, src0, C0, src1, C1, N, H, W, wgt, Cout, scale, shift, relu, out, stream);
  TapGeom g;
  geom_conv3x3(g, N, H, W);
  g.f16 = 0;
  TcStats stt = {sums_q, 0};
  const int rc = run_tc_fwd(g, src0, C0, src1, C1, wgt, Cout, out, scale, shift, relu, 0, (cudaStream_t)stream, nullptr, &stt);
  *stats_done = stt.done;
  return rc;
}

extern "C" int dcb_convT2x2_fwd_stats(int dtype, const void* src, int Cin, int N, int h, int w, const void* wgt, int Cout,
                                      const float* scale, const float* shift, int relu, void* out, long long* sums_q,
                                      int* stats_done, dcb_stream_t stream) {
  DCB_CHECK_ARG(src && wgt && out && sums_q && stats_done && N > 0 && h > 0 && w > 0 && Cin > 0 && Cout > 0,
                "dcb_convT2x2_fwd_stats: bad arguments");
  *stats_done = 0;
  if (dtype != DCB_BF16) return dcb_convT2x2_fwd(dtype, src, Cin, N, h, w, wgt, Cout, scale, shift, relu, out, stream);
  TapGeom g;
  geom_convT_fwd(g, N, h, w);
  g.f16 = 0;
  TcStats stt = {sums_q, 0};
  const int rc = run_tc_fwd(g, src, Cin, nullptr, 0, wgt, Cout, out, scale, shift, relu, 0, (cudaStream_t)stream, nullptr, &stt);
  *stats_done = stt.done;
  return rc;
}

extern "C" int dcb_conv3x3_dgrad(int dtype, const void* dy, int Cout, int N, int H, int W, const void* wgt_dgrad, int Cin,
                                 float* dx, dcb_stream_t stream) {
  DCB_CHECK_ARG(dy && wgt_dgrad && dx && N > 0 && H > 0 && W > 0 && Cin > 0 && Cout > 0, "dcb_conv3x3_dgrad: bad arguments");
  TapGeom g;
  geom_conv3x3(g, N, H, W);
  g.f16 = (dtype == DCB_F16);
  if (dtype == DCB_F32)
    return run_f32_fwd(g, (const float*)dy, Cout, nullptr, 0, (const float*)wgt_dgrad, Cin, dx, nullptr, nullptr, 0,
                       (cudaStream_t)stream);
  if (dtype == DCB_BF16 || dtype == DCB_F16)
    return run_tc_fwd(g, dy, Cout, nullptr, 0, wgt_dgrad, Cin, dx, nullptr, nullptr, 0, 1, (cudaStream_t)stream);
  return fail(DCB_ERR_INVALID_ARGUMENT, "unknown dtype %d", dtype);
}

extern "C" int dcb_convT2x2_fwd(int dtype, const void* src, int Cin, int N, int h, int w, const void* wgt, int Cout,
                                const float* scale, const float* shift, int relu, void* out, dcb_stream_t stream) {
  DCB_CHECK_ARG(src && wgt && out && N > 0 && h > 0 && w > 0 && Cin > 0 && Cout > 0, "dcb_convT2x2_fwd: bad arguments");
  TapGeom g;
  geom_convT_fwd(g, N, h, w);
  g.f16 = (dtype == DCB_F16);
  if (dtype == DCB_F32)
    return run_f32_fwd(g, (const float*)src, Cin, nullptr, 0, (const float*)wgt, Cout, (float*)out, scale, shift, relu,
                       (cudaStream_t)stream);
  if (dtype == DCB_BF16 || dtype == DCB_F16)
    return run_tc_fwd(g, src, Cin, nullptr, 0, wgt, Cout, out, scale, shift, relu, 0, (cudaStream_t)stream);
  return fail(DCB_ERR_INVALID_ARGUMENT, "unknown dtype %d", dtype);
}

extern "C" int dcb_convT2x2_dgrad(int dtype, const void* dy, int Cout, int N, int h, int w, const void* wgt, int Cin,
                                  float* dx, dcb_stream_t stream) {
  DCB_CHECK_ARG(dy && wgt && dx && N > 0 && h > 0 && w > 0 && Cin > 0 && Cout > 0, "dcb_convT2x2_dgrad: bad arguments");
  TapGeom g;
  geom_convT_dgrad(g, N, h, w);
  g.f16 = (dtype == DCB_F16);
  if (dtype == DCB_F32)
    return run_f32_fwd(g, (const float*)dy, Cout, nullptr, 0, (const float*)wgt, Cin, dx, nullptr, nullptr, 0,
                       (cudaStream_t)stream);
  if (dtype == DCB_BF16 || dtype == DCB_F16)
    return run_tc_fwd(g, dy, Cout, nullptr, 0, wgt, Cin, dx, nullptr, nullptr, 0, 1, (cudaStream_t)stream);
  return fail(DCB_ERR_INVALID_ARGUMENT, "unknown dtype %d", dtype);
}

extern "C" int dcb_conv3x3_wgrad_workspace_bytes(int dtype, int N, int H, int W, int Cin, int Cout, size_t* bytes) {
  DCB_CHECK_ARG(bytes && N > 0 && H > 0 && W > 0 && Cin > 0 && Cout > 0, "dcb_conv3x3_wgrad_workspace_bytes: bad arguments");
  TapGeom g;
  geom_conv3x3(g, N, H, W);
  g.f16 = (dtype == DCB_F16);
  if (dtype == DCB_F32) *bytes = (size_t)f32_wgrad_splits(g, Cin, Cout) * 9 * Cin * Cout * sizeof(float);
  else *bytes = tc_wgrad_workspace(g, Cin, Cout);
  return DCB_OK;
}

extern "C" int dcb_conv3x3_wgrad(int dtype, const void* src0, int C0, const void* src1, int C1, int N, int H, int W,
                                 const void* dy, int Cout, float* dW, void* ws, size_t ws_bytes, dcb_stream_t stream) {
  DCB_CHECK_ARG(src0 && dy && dW && N > 0 && H > 0 && W > 0 && C0 > 0 && C1 >= 0 && Cout > 0 && (C1 == 0 || src1),
                "dcb_conv3x3_wgrad: bad arguments");
  TapGeom g;
  geom_conv3x3(g, N, H, W);
  g.f16 = (dtype == DCB_F16);
  if (dtype == DCB_F32)
    return run_f32_wgrad(g, (const float*)src0, C0, (const float*)src1, C1, (const float*)dy, Cout, dW, ws, ws_bytes,
                         (cudaStream_t)stream);
  if (dtype == DCB_BF16 || dtype == DCB_F16) return run_tc_wgrad(g, src0, C0, src1, C1, dy, Cout, dW, ws, ws_bytes, (cudaStream_t)stream);
  return fail(DCB_ERR_INVALID_ARGUMENT, "unknown dtype %d", dtype);
}

extern "C" int dcb_convT2x2_wgrad_workspace_bytes(int dtype, int N, int h, int w, int Cin, int Cout, size_t* bytes) {
  DCB_CHECK_ARG(bytes && N > 0 && h > 0 && w > 0 && Cin > 0 && Cout > 0, "dcb_convT2x2_wgrad_workspace_bytes: bad arguments");
  TapGeom g;
  geom_convT_dgrad(g, N, h, w);
  g.f16 = (dtype == DCB_F16);
  if (dtype == DCB_F32) *bytes = (size_t)f32_wgrad_splits(g, Cout, Cin) * 4 * Cin * Cout * sizeof(float);
  else *bytes = tc_wgrad_workspace(g, Cout, Cin);
  return DCB_OK;
}

// dW[a,b][co][ci] = sum_{n,i,j} dy[n,2i+a,2j+b,co] * x[n,i,j,ci]: the gathered operand is dy, the
// per-position operand is x
extern "C" int dcb_convT2x2_wgrad(int dtype, const void* x, int Cin, int N, int h, int w, const void* dy, int Cout,
                                  float* dW, void* ws, size_t ws_bytes, dcb_stream_t stream) {
  DCB_CHECK_ARG(x && dy && dW && N > 0 && h > 0 && w > 0 && Cin > 0 && Cout > 0, "dcb_convT2x2_wgrad: bad arguments");
  TapGeom g;
  geom_convT_dgrad(g, N, h, w);
  g.f16 = (dtype == DCB_F16);
  if (dtype == DCB_F32)
    return run_f32_wgrad(g, (const float*)dy, Cout, nullptr, 0, (const float*)x, Cin, dW, ws, ws_bytes,
                         (cudaStream_t)stream);
  if (dtype == DCB_BF16 || dtype == DCB_F16) return run_tc_wgrad(g, dy, Cout, nullptr, 0, x, Cin, dW, ws, ws_bytes, (cudaStream_t)stream);
  return fail(DCB_ERR_INVALID_ARGUMENT, "unknown dtype %d", dtype);
}
