// Small device helpers shared by the memory-bound kernels.
#pragma once
#include "common.cuh"

namespace dcb {

template <typename T> __device__ __forceinline__ float4 load4(const T* p);
template <> __device__ __forceinline__ float4 load4<float>(const float* p) {
  return *reinterpret_cast<const float4*>(p);
}
template <> __device__ __forceinline__ float4 load4<__nv_bfloat16>(const __nv_bfloat16* p) {
  uint2 u = *reinterpret_cast<const uint2*>(p);
  __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&u.x);
  __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&u.y);
  float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
  return make_float4(fa.x, fa.y, fb.x, fb.y);
}
template <> __device__ __forceinline__ float4 load4<__half>(const __half* p) {
  uint2 u = *reinterpret_cast<const uint2*>(p);
  const float2 fa = __half22float2(*reinterpret_cast<__half2*>(&u.x)), fb = __half22float2(*reinterpret_cast<__half2*>(&u.y));
  return make_float4(fa.x, fa.y, fb.x, fb.y);
}
template <typename T> __device__ __forceinline__ void store4(T* p, float4 v);
template <> __device__ __forceinline__ void store4<__half>(__half* p, float4 v) {
  __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
  uint2 u;
  u.x = *reinterpret_cast<uint32_t*>(&a);
  u.y = *reinterpret_cast<uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p) = u;
}
template <> __device__ __forceinline__ void store4<float>(float* p, float4 v) {
  *reinterpret_cast<float4*>(p) = v;
}
template <> __device__ __forceinline__ void store4<__nv_bfloat16>(__nv_bfloat16* p, float4 v) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
  uint2 u;
  u.x = *reinterpret_cast<uint32_t*>(&a);
  u.y = *reinterpret_cast<uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p) = u;
}

// 8 consecutive channels (16 bytes of bf16 / 32 bytes of fp32)
template <typename T> __device__ __forceinline__ void load8(const T* p, float (&v)[8]);
template <> __device__ __forceinline__ void load8<float>(const float* p, float (&v)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
template <> __device__ __forceinline__ void load8<__nv_bfloat16>(const __nv_bfloat16* p, float (&v)[8]) {
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[i]));
    v[2 * i] = f.x; v[2 * i + 1] = f.y;
  }
}

template <> __device__ __forceinline__ void load8<__half>(const __half* p, float (&v)[8]) {
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
    v[2 * i] = f.x; v[2 * i + 1] = f.y;
  }
}
template <typename T> __device__ __forceinline__ void store8(T* p, const float (&v)[8]);
template <> __device__ __forceinline__ void store8<__half>(__half* p, const float (&v)[8]) {
  uint32_t w[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __half2 b = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
    w[i] = *reinterpret_cast<uint32_t*>(&b);
  }
  *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
}
template <> __device__ __forceinline__ void store8<float>(float* p, const float (&v)[8]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
template <> __device__ __forceinline__ void store8<__nv_bfloat16>(__nv_bfloat16* p, const float (&v)[8]) {
  uint32_t w[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __nv_bfloat162 b = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    w[i] = *reinterpret_cast<uint32_t*>(&b);
  }
  *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
}
template <typename T, int VEC> __device__ __forceinline__ void storev(T* p, const float (&v)[VEC]) {
  if constexpr (VEC == 8) store8<T>(p, v);
  else store4<T>(p, make_float4(v[0], v[1], v[2], v[3]));
}

template <typename T, int VEC> __device__ __forceinline__ void loadv(const T* p, float (&v)[VEC]) {
  if constexpr (VEC == 8) {
    load8<T>(p, v);
  } else {
    const float4 a = load4<T>(p);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
  }
}

// np.pad(mode='reflect'), extended to negative i.  For pads longer than the axis np.pad reflects repeatedly, which is
// this periodic map.
__device__ __forceinline__ int reflect_index(int i, int n) {
  if (n == 1) return 0;
  const int period = 2 * (n - 1);
  int r = (i < 0 ? -i : i) % period;
  return r < n ? r : period - r;
}

// packed fp32x2 FMA (sm_100): d = a * b + c on two values at once, one issue slot
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  uint64_t ua, ub, uc, ud;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ua) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(ub) : "f"(b.x), "f"(b.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(uc) : "f"(c.x), "f"(c.y));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(ud) : "l"(ua), "l"(ub), "l"(uc));
  float2 d;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(ud));
  return d;
}

// Philox4x32-10 counter-based RNG (Salmon et al. 2011); one call -> 4 x uint32.
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0; key.y += W1;
  }
  return ctr;
}

// Dropout keep-mask: element e draws a 16-bit uniform - half-word (e % 8) of Philox4x32-10(counter = e / 8, key = seed,
// extra counter word = layer id) - and is kept when it is >= floor(p_drop * 65536); kept elements are scaled by
// 1 / (1 - p_drop).  One Philox call therefore serves 8 consecutive elements (one 16-byte bf16 vector): the 7 dropout
// layers of a training step were issue bound on the generator when it served only 4 (32-bit uniforms).
__device__ __forceinline__ void dropout_scale8(unsigned long long seed, uint32_t layer, unsigned long long idx8, float p_drop,
                                               float (&k)[8]) {
  const uint4 r = philox4x32_10(make_uint4((uint32_t)idx8, (uint32_t)(idx8 >> 32), layer, 0u),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const float inv = 1.f / (1.f - p_drop);
  const uint32_t thr = (uint32_t)(p_drop * 65536.f);
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    k[2 * i] = (w[i] & 0xffffu) >= thr ? inv : 0.f;
    k[2 * i + 1] = (w[i] >> 16) >= thr ? inv : 0.f;
  }
}
// 4 consecutive elements starting at flat index idx4 * 4 (the lower or upper half of their group of 8)
__device__ __forceinline__ float4 dropout_scale4(unsigned long long seed, uint32_t layer, unsigned long long idx4,
                                                 float p_drop) {
  float k[8];
  dropout_scale8(seed, layer, idx4 >> 1, p_drop, k);
  return (idx4 & 1ull) ? make_float4(k[4], k[5], k[6], k[7]) : make_float4(k[0], k[1], k[2], k[3]);
}

}  // namespace dcb
