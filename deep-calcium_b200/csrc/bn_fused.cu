// Training-mode BatchNorm of the UNet2DS blocks (Keras 2.0.6 BatchNormalization, unet_2d_summary.py:157,165) as
// SINGLE-LAUNCH kernels: batch statistics are a grid-wide dependency, so the separate-pass version costs four launches
// per layer (stats, finalize+apply, backward reduce, backward apply: 88 launches and ~40 % of a 32-crop training step).
// Here one persistent kernel does   reduce -> cross-CTA total -> grid barrier -> apply,
// re-reading in the second phase what the first phase just pulled through L2 (every tensor of a 128^2 x 32 step is
// smaller than the 126 MB L2).  The cross-CTA total is a sum of 64-bit FIXED-POINT integers (per-CTA fp64 partials in a
// fixed order, integer atomics across CTAs), so results are bit-reproducible run to run - no floating-point atomics.
//
// Data-parallel training (SyncBN, SURVEY 8e): with `peers` set, the per-channel totals of every rank are exchanged
// INSIDE the kernel over NVLink - each rank stores its totals into every peer's exchange slot (peer-mapped memory),
// publishes a flag carrying the step number, waits for the peers' flags and adds the slots in rank order - instead of
// an NCCL all-reduce between two launches.
#include <cooperative_groups.h>
#include <type_traits>
#include "elementwise.cuh"
#include "stats_epilogue.cuh"

namespace dcb {

struct PeerView {
  int world, rank;
  double* xchg[8];              // peer p's exchange area (peer-mapped): [slot][rank][2 * C] doubles
  unsigned long long* flags[8]; // peer p's flag area: [slot][rank]
  long long slot_doubles;       // offset of this call's slot inside the exchange area, in doubles
  int slot_flag;                // index of this call's slot inside the flag area (x 8 ranks)
  const unsigned long long* epoch;   // device counter that differs between consecutive steps (dcb_step_advance state)
};

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// All CTAs of the grid are co-resident (the host sizes the grid from the occupancy query).  `counter` starts at 0
// (the caller zeroes the sync words before the launch).  A protocol failure traps after ~2 s instead of hanging.
__device__ __forceinline__ void grid_barrier(unsigned* counter) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(counter, 1u);
    const long long t0 = clock64();
    while (ld_acquire_u32(counter) < gridDim.x) {
      __nanosleep(64);
      if (clock64() - t0 > 4000000000LL) __trap();
    }
    __threadfence();
  }
  __syncthreads();
}

// Cross-CTA totals as 64-bit FIXED-POINT integer atomics (the caller zeroes totals_q): integer addition is associative, so
// the total does not depend on the arrival order - bit-reproducible like a fixed-order tree, but it needs neither
// the workspace round trip of the per-CTA partials nor the second grid barrier.  Units: 2^-20 for the forward sums of
// activations (range 8.8e12), 2^-40 for the backward sums of gradients (range 8.4e6, resolution 9e-13).
constexpr double FWD_UNITS_INV = 1048576.0, FWD_UNITS = 1.0 / 1048576.0;                 // 2^20
constexpr double BWD_UNITS_INV = 1099511627776.0, BWD_UNITS = 1.0 / 1099511627776.0;     // 2^40
// The backward sums (sum dz, sum dz * xhat) cancel to ~1e-3 of their terms in this network, so ANY change in how fp32
// partial sums are grouped (CTA partition, batch split over ranks, kernel variant) showed up as 1e-3 .. 5e-3 relative
// differences in the beta / gamma gradients.  They are therefore accumulated EXACTLY: every element is converted to 2^-40
// fixed point (one fp32 multiply by a power of two - exact - and one round-to-integer, the same for an element wherever
// it is processed) and all additions are 64-bit integer additions: the totals are independent of thread / CTA / rank
// partition and of the order of arrival, bit for bit.
__device__ __forceinline__ long long to_q40(float v) { return __float2ll_rn(v * 1099511627776.f); }
// The 64-bit conversions cost the 16-bit training mode 6 % of its step (16 per row and thread in a memory-bound kernel),
// where the comparison between two runs is at 16-bit tolerance anyway: EXACT per-element accumulation in the fp32 check
// mode (the mode parity is judged in), fp32 per-thread partials converted once per thread otherwise - the sums across
// threads / CTAs / ranks are integer sums in both.
__device__ __forceinline__ long long to_q20(float v) { return __float2ll_rn(v * 1048576.f); }
template <bool EXACT, bool Q40> struct FixAcc;
template <bool Q40> struct FixAcc<true, Q40> {
  long long v = 0;
  __device__ __forceinline__ void add(float x) { v += Q40 ? to_q40(x) : to_q20(x); }
  __device__ __forceinline__ long long fixed() const { return v; }
};
template <bool Q40> struct FixAcc<false, Q40> {
  float v = 0.f;
  __device__ __forceinline__ void add(float x) { v += x; }
  __device__ __forceinline__ long long fixed() const { return Q40 ? to_q40(v) : to_q20(v); }
};
template <bool EXACT> using BwdAcc = FixAcc<EXACT, true>;    // gradient sums, 2^-40 units
template <bool EXACT> using FwdAcc = FixAcc<EXACT, false>;   // activation sums, 2^-20 units (the forward statistics of the check
                                                             // mode are exact for the same reason: partition-independent)

// The totals live in the caller's workspace, which is ZERO when a launch starts: after every CTA has taken its copy, the
// last one to say so (second sync word) clears them again for the next launch that uses the workspace.
__device__ __forceinline__ void release_totals(long long* totals_q, int V, unsigned* done_counter) {
  __shared__ int s_last_reader;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    s_last_reader = (atomicAdd(done_counter, 1u) == gridDim.x - 1) ? 1 : 0;
  }
  __syncthreads();
  if (s_last_reader)
    for (int i = threadIdx.x; i < V; i += blockDim.x) totals_q[i] = 0;
}

// SyncBN exchange of the V local totals (see the file comment).  Returns with s_tot[0..V) = sum over ranks.
template <typename GetFn>
__device__ __forceinline__ void peer_exchange_fn(const PeerView& pv, GetFn get, int V, double* s_tot) {
  const unsigned long long epoch = *pv.epoch;
  if (blockIdx.x == 0) {
    for (int p = 0; p < pv.world; ++p) {
      double* dst = pv.xchg[p] + pv.slot_doubles + (long long)pv.rank * V;
      for (int i = threadIdx.x; i < V; i += blockDim.x) dst[i] = get(i);
    }
    __threadfence_system();
    __syncthreads();
    if ((int)threadIdx.x < pv.world) st_release_sys_u64(pv.flags[threadIdx.x] + pv.slot_flag * 8 + pv.rank, epoch);
  }
  if ((int)threadIdx.x < pv.world) {
    const unsigned long long* f = pv.flags[pv.rank] + pv.slot_flag * 8 + threadIdx.x;
    const long long t0 = clock64();
    while (ld_acquire_sys_u64(f) != epoch) {
      __nanosleep(128);
      if (clock64() - t0 > 20000000000LL) __trap();
    }
  }
  __syncthreads();
  const double* src = pv.xchg[pv.rank] + pv.slot_doubles;
  for (int i = threadIdx.x; i < V; i += blockDim.x) {
    double acc = 0;
    for (int r = 0; r < pv.world; ++r) acc += __ldcv(src + (long long)r * V + i);
    s_tot[i] = acc;
  }
  __syncthreads();
}

__device__ __forceinline__ void peer_exchange(const PeerView& pv, const double* __restrict__ totals, int V, double* s_tot) {
  peer_exchange_fn(pv, [&](int i) { return __ldcg(totals + i); }, V, s_tot);
}

struct BnFwdParams {
  const void* x; void* y; void* pool;   // raw conv output [M][C], activation out, optional 2x2 max-pooled copy
  long long M, M_total; int C;
  int N, H, W;                          // pixel grid (pooling only)
  const float* gamma; const float* beta; float eps, momentum;
  float* moving_mean; float* moving_var; float* scale; float* shift; float* mean; float* rstd;
  int relu; float p_drop; unsigned long long seed; const unsigned long long* seed_dev; unsigned layer;
  double* totals; unsigned* sync;           // totals: 64-bit fixed-point integers (2 * C), zero on entry
  const long long* sums_q;              // PRE instantiation: fixed-point batch sums of a conv epilogue (stats_epilogue.cuh)
  PeerView pv;
};

// PRE: the batch sums are already in p.totals (taken by the conv epilogue that produced x, stats_epilogue.cuh): phase 1
// and both grid barriers disappear, the grid needs no co-residency
template <typename T, int VEC, bool POOL, bool PRE = false>
__global__ void __launch_bounds__(256)
bn_train_fwd_kernel(const BnFwdParams p) {
  extern __shared__ double s_dyn[];
  if (threadIdx.x == 0) pdl_trigger();     // programmatic dependent launch: the grid is resident when the producer finishes
  pdl_wait();
  const int C = p.C, V = 2 * C;
  const T* __restrict__ x = reinterpret_cast<const T*>(p.x);
  const int lanes_c = C / VEC, rows_par = 256 / lanes_c;
  const int tc = threadIdx.x % lanes_c, tr = threadIdx.x / lanes_c;
  const long long rows_per_cta = (p.M + gridDim.x - 1) / gridDim.x;
  const long long r0 = (long long)blockIdx.x * rows_per_cta;
  long long r1 = r0 + rows_per_cta; if (r1 > p.M) r1 = p.M;
  // ---------------- phase 1: per-CTA partial sums of x and x^2
  if constexpr (!PRE) {
    FwdAcc<std::is_same<T, float>::value> s[VEC], q[VEC];
    const T* base = x + tc * VEC;
    long long r = r0 + tr;
    for (; r + 3LL * rows_par < r1; r += 4LL * rows_par) {
      float v[4][VEC];
#pragma unroll
      for (int u = 0; u < 4; ++u) loadv<T, VEC>(base + (r + (long long)u * rows_par) * C, v[u]);
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int i = 0; i < VEC; ++i) { s[i].add(v[u][i]); q[i].add(v[u][i] * v[u][i]); }
    }
    for (; r < r1; r += rows_par) {
      float v[VEC];
      loadv<T, VEC>(base + r * C, v);
#pragma unroll
      for (int i = 0; i < VEC; ++i) { s[i].add(v[i]); q[i].add(v[i] * v[i]); }
    }
    long long* sh = reinterpret_cast<long long*>(s_dyn);      // 256 * 2 * VEC int64
#pragma unroll
    for (int i = 0; i < VEC; ++i) { sh[threadIdx.x * 2 * VEC + i] = s[i].fixed(); sh[threadIdx.x * 2 * VEC + VEC + i] = q[i].fixed(); }
    __syncthreads();
    for (int idx = threadIdx.x; idx < lanes_c * 2 * VEC; idx += 256) {
      const int lc = idx / (2 * VEC), comp = idx % (2 * VEC);
      long long acc = 0;
      for (int rr = 0; rr < rows_par; ++rr) acc += sh[(rr * lanes_c + lc) * 2 * VEC + comp];
      atomicAdd(reinterpret_cast<unsigned long long*>(p.totals) + (comp / VEC) * C + lc * VEC + (comp % VEC), (unsigned long long)acc);
    }
    grid_barrier(p.sync + 0);
  }
  // ---------------- per-channel coefficients (every CTA; block 0 publishes them and updates the moving statistics)
  double* s_tot = s_dyn;                               // V doubles
  float* s_sc = reinterpret_cast<float*>(s_dyn + V); float* s_sh = s_sc + C;
  if constexpr (PRE) {
    if (p.pv.world > 1) {
      peer_exchange_fn(p.pv, [&](int i) { return (double)__ldcg(p.sums_q + i) * tc::STATS_Q_INV; }, V, s_tot);
    } else {
      for (int i = threadIdx.x; i < V; i += blockDim.x) s_tot[i] = (double)__ldcg(p.sums_q + i) * tc::STATS_Q_INV;
      __syncthreads();
    }
  } else {
    const long long* tq = reinterpret_cast<const long long*>(p.totals);
    if (p.pv.world > 1) {
      peer_exchange_fn(p.pv, [&](int i) { return (double)__ldcg(tq + i) * FWD_UNITS; }, V, s_tot);
    } else {
      for (int i = threadIdx.x; i < V; i += blockDim.x) s_tot[i] = (double)__ldcg(tq + i) * FWD_UNITS;
      __syncthreads();
    }
    release_totals(reinterpret_cast<long long*>(p.totals), V, p.sync + 1);
  }
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const double mean = s_tot[c] / (double)p.M_total;
    double var = s_tot[C + c] / (double)p.M_total - mean * mean;
    if (var < 0) var = 0;
    const float rstd = (float)(1.0 / sqrt(var + (double)p.eps));
    const float sc = p.gamma[c] * rstd;
    const float shv = p.beta[c] - (float)mean * sc;
    s_sc[c] = sc; s_sh[c] = shv;
    if (blockIdx.x == 0) {
      p.scale[c] = sc; p.shift[c] = shv; p.mean[c] = (float)mean; p.rstd[c] = rstd;
      if (p.moving_mean) {   // Keras: moving <- moving*m + batch*(1-m), biased batch variance
        p.moving_mean[c] = p.moving_mean[c] * p.momentum + (float)mean * (1.f - p.momentum);
        p.moving_var[c] = p.moving_var[c] * p.momentum + (float)var * (1.f - p.momentum);
      }
    }
  }
  __syncthreads();
  // ---------------- phase 2: y = relu(x * scale + shift) (* dropout keep mask) [, 2x2 max-pool]
  unsigned long long seed = p.seed;
  if (p.seed_dev) seed ^= *p.seed_dev;
  T* __restrict__ y = reinterpret_cast<T*>(p.y);
  auto apply = [&](long long i, float (&v)[VEC]) {      // i = index of the VEC-channel group in the flat tensor
    const int c = (int)((i * VEC) % C);
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      v[j] = fmaf(v[j], s_sc[c + j], s_sh[c + j]);
      if (p.relu) v[j] = fmaxf(v[j], 0.f);
    }
    if (p.p_drop > 0.f) {
#pragma unroll
      for (int h = 0; h < VEC / 4; ++h) {
        const float4 k = dropout_scale4(seed, p.layer, (unsigned long long)(i * (VEC / 4) + h), p.p_drop);
        v[4 * h] *= k.x; v[4 * h + 1] *= k.y; v[4 * h + 2] *= k.z; v[4 * h + 3] *= k.w;
      }
    }
  };
  if constexpr (!POOL) {
    // the CTA re-reads its own rows (what phase 1 just pulled through L2)
    const long long i0 = r0 * lanes_c, i1 = r1 * lanes_c;
    long long i = i0 + threadIdx.x;
    for (; i + 3 * 256 < i1; i += 4 * 256) {            // four independent 16-byte loads in flight per thread
      float v[4][VEC];
#pragma unroll
      for (int u = 0; u < 4; ++u) loadv<T, VEC>(x + (i + u * 256) * VEC, v[u]);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        apply(i + u * 256, v[u]);
        storev<T, VEC>(y + (i + u * 256) * VEC, v[u]);
      }
    }
    for (; i < i1; i += 256) {
      float v[VEC];
      loadv<T, VEC>(x + i * VEC, v);
      apply(i, v);
      storev<T, VEC>(y + i * VEC, v);
    }
  } else {
    T* __restrict__ pool = reinterpret_cast<T*>(p.pool);
    const int OH = p.H / 2, OW = p.W / 2;
    const long long nq = (long long)p.N * OH * OW * lanes_c;
    for (long long qd = (long long)blockIdx.x * 256 + threadIdx.x; qd < nq; qd += (long long)gridDim.x * 256) {
      long long t = qd;
      const int lc = (int)(t % lanes_c); t /= lanes_c;
      const int ow = (int)(t % OW); t /= OW;
      const int oh = (int)(t % OH); const int n = (int)(t / OH);
      const long long pix00 = ((long long)n * p.H + 2 * oh) * p.W + 2 * ow;
      float m[VEC];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const long long pix = pix00 + (k >> 1) * p.W + (k & 1);
        const long long i = pix * lanes_c + lc;
        float v[VEC];
        loadv<T, VEC>(x + i * VEC, v);
        apply(i, v);
        storev<T, VEC>(y + i * VEC, v);
        // pooling compares the STORED (rounded) activations, like the standalone kernel that reads them back
        float rv[VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) rv[j] = to_f32<T>(from_f32<T>(v[j]));
#pragma unroll
        for (int j = 0; j < VEC; ++j) m[j] = k == 0 ? rv[j] : fmaxf(m[j], rv[j]);
      }
      storev<T, VEC>(pool + qd * VEC, m);
    }
  }
}

struct BnBwdParams {
  const float* dy; int ldy, offy;       // upstream gradient (fp32 view: row stride ldy, channel offset offy)
  const float* gpix; const float* wd;   // or (gpix != null) the rank-1 gradient of the softmax head: dy[r][c] = gpix[r] * wd[c]
  const void* x; void* draw;            // raw conv output [M][C]; gradient w.r.t. it (may alias x)
  long long M, M_total; int C;
  const float* scale; const float* shift; const float* mean; const float* rstd;
  float p_drop; unsigned long long seed; const unsigned long long* seed_dev; unsigned layer;
  float dgb_scale; float* dgamma; float* dbeta;
  double* totals; unsigned* sync;           // totals: 64-bit fixed-point integers (2 * C), zero on entry
  PeerView pv;
};

// dz = dY * keepscale * [x*scale+shift > 0];  totals[c] = sum dz, totals[C+c] = sum dz * xhat;
// d_raw = scale * (dz - mean(dz) - xhat * mean(dz*xhat)) = scale*dz + k1*(x - mean) + k0
template <typename T, int VEC>
__global__ void __launch_bounds__(256)
bn_train_bwd_kernel(const BnBwdParams p) {
  extern __shared__ double s_dyn[];
  if (threadIdx.x == 0) pdl_trigger();
  pdl_wait();
  const int C = p.C, V = 2 * C;
  const T* __restrict__ x = reinterpret_cast<const T*>(p.x);
  unsigned long long seed = p.seed;
  if (p.seed_dev) seed ^= *p.seed_dev;
  const int lanes_c = C / VEC, rows_par = 256 / lanes_c;
  const int tc = threadIdx.x % lanes_c, tr = threadIdx.x / lanes_c;
  const long long rows_per_cta = (p.M + gridDim.x - 1) / gridDim.x;
  const long long r0 = (long long)blockIdx.x * rows_per_cta;
  long long r1 = r0 + rows_per_cta; if (r1 > p.M) r1 = p.M;
  const int c = tc * VEC;
  float sc[VEC], sh[VEC], mu[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) { sc[i] = p.scale[c + i]; sh[i] = p.shift[c + i]; mu[i] = p.mean[c + i]; }
  auto masked = [&](long long r, float (&g)[VEC], const float (&v)[VEC]) {
    if (p.p_drop > 0.f) {
      if constexpr (VEC == 8) {
        float k[8];
        dropout_scale8(seed, p.layer, (unsigned long long)((r * C + c) >> 3), p.p_drop, k);
#pragma unroll
        for (int i = 0; i < 8; ++i) g[i] *= k[i];
      } else {
        const float4 k0 = dropout_scale4(seed, p.layer, (unsigned long long)((r * C + c) >> 2), p.p_drop);
        g[0] *= k0.x; g[1] *= k0.y; g[2] *= k0.z; g[3] *= k0.w;
      }
    }
#pragma unroll
    for (int i = 0; i < VEC; ++i)
      if (fmaf(v[i], sc[i], sh[i]) <= 0.f) g[i] = 0.f;
  };
  float wdv[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) wdv[i] = p.gpix ? p.wd[c + i] : 0.f;
  auto load_dy = [&](long long r, float (&g)[VEC]) {
    if (p.gpix) {
      const float gp = p.gpix[r];
#pragma unroll
      for (int i = 0; i < VEC; ++i) g[i] = gp * wdv[i];
    } else {
      loadv<float, VEC>(p.dy + r * p.ldy + p.offy + c, g);
    }
  };
  // ---------------- phase 1: exact fixed-point sums (see to_q40)
  {
    float rs[VEC];
    BwdAcc<std::is_same<T, float>::value> s[VEC], q[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) rs[i] = p.rstd[c + i];
    auto accumulate = [&](long long r, float (&g)[VEC], const float (&v)[VEC]) {
      masked(r, g, v);
#pragma unroll
      for (int i = 0; i < VEC; ++i) { s[i].add(g[i]); q[i].add(g[i] * ((v[i] - mu[i]) * rs[i])); }
    };
    long long r = r0 + tr;
    for (; r + rows_par < r1; r += 2LL * rows_par) {
      float g0[VEC], g1[VEC], v0[VEC], v1[VEC];
      load_dy(r, g0);
      load_dy(r + rows_par, g1);
      loadv<T, VEC>(x + r * C + c, v0);
      loadv<T, VEC>(x + (r + rows_par) * C + c, v1);
      accumulate(r, g0, v0);
      accumulate(r + rows_par, g1, v1);
    }
    for (; r < r1; r += rows_par) {
      float g0[VEC], v0[VEC];
      load_dy(r, g0);
      loadv<T, VEC>(x + r * C + c, v0);
      accumulate(r, g0, v0);
    }
    long long* shm = reinterpret_cast<long long*>(s_dyn);      // 256 * 2 * VEC int64
#pragma unroll
    for (int i = 0; i < VEC; ++i) { shm[threadIdx.x * 2 * VEC + i] = s[i].fixed(); shm[threadIdx.x * 2 * VEC + VEC + i] = q[i].fixed(); }
    __syncthreads();
    for (int idx = threadIdx.x; idx < lanes_c * 2 * VEC; idx += 256) {
      const int lc = idx / (2 * VEC), comp = idx % (2 * VEC);
      long long acc = 0;
      for (int rr = 0; rr < rows_par; ++rr) acc += shm[(rr * lanes_c + lc) * 2 * VEC + comp];
      atomicAdd(reinterpret_cast<unsigned long long*>(p.totals) + (comp / VEC) * C + lc * VEC + (comp % VEC), (unsigned long long)acc);
    }
  }
  grid_barrier(p.sync + 0);
  double* s_tot = s_dyn;
  {
    const long long* tq = reinterpret_cast<const long long*>(p.totals);
    if (p.pv.world > 1) {
      peer_exchange_fn(p.pv, [&](int i) { return (double)__ldcg(tq + i) * BWD_UNITS; }, V, s_tot);
    } else {
      for (int i = threadIdx.x; i < V; i += blockDim.x) s_tot[i] = (double)__ldcg(tq + i) * BWD_UNITS;
      __syncthreads();
    }
    release_totals(reinterpret_cast<long long*>(p.totals), V, p.sync + 1);
  }
  // ---------------- phase 2: this thread's channels only (same row partition as phase 1)
  float k1[VEC], k0[VEC];
  {
    const double invM = 1.0 / (double)p.M_total;
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const double scd = (double)sc[i], m1 = s_tot[c + i] * invM, m2 = s_tot[C + c + i] * invM;
      k1[i] = (float)(-scd * (double)p.rstd[c + i] * m2);
      k0[i] = (float)(-scd * m1);
    }
  }
  if (blockIdx.x == 0) {
    for (int cc = threadIdx.x; cc < C; cc += blockDim.x) {
      if (p.dbeta) p.dbeta[cc] = (float)(s_tot[cc] * (double)p.dgb_scale);
      if (p.dgamma) p.dgamma[cc] = (float)(s_tot[C + cc] * (double)p.dgb_scale);
    }
  }
  T* __restrict__ draw = reinterpret_cast<T*>(p.draw);
  // The rows are walked BACKWARDS: phase 1 went through this CTA's range in ascending order, so its tail is what the L2
  // still holds (dy + x of a full-resolution layer are 100 MB); an ascending second pass would start with the rows that
  // were evicted first and push the resident ones out before reaching them.
  const long long first = r0 + tr;
  long long nrows = first < r1 ? (r1 - first + rows_par - 1) / rows_par : 0;
  long long r = first + (nrows - 1) * rows_par;          // this thread's last row
  for (; nrows >= 2; nrows -= 2, r -= 2LL * rows_par) {   // two rows (2 x 48 bytes of loads) in flight per thread
    float g0[VEC], g1[VEC], v0[VEC], v1[VEC], o[VEC];
    const long long ra = r, rb = r - rows_par;
    load_dy(ra, g0);
    load_dy(rb, g1);
    loadv<T, VEC>(x + ra * C + c, v0);
    loadv<T, VEC>(x + rb * C + c, v1);
    masked(ra, g0, v0);
    masked(rb, g1, v1);
#pragma unroll
    for (int j = 0; j < VEC; ++j) o[j] = fmaf(sc[j], g0[j], fmaf(k1[j], v0[j] - mu[j], k0[j]));
    storev<T, VEC>(draw + ra * C + c, o);
#pragma unroll
    for (int j = 0; j < VEC; ++j) o[j] = fmaf(sc[j], g1[j], fmaf(k1[j], v1[j] - mu[j], k0[j]));
    storev<T, VEC>(draw + rb * C + c, o);
  }
  if (nrows == 1) {
    float g[VEC], v[VEC], o[VEC];
    load_dy(r, g);
    loadv<T, VEC>(x + r * C + c, v);
    masked(r, g, v);
#pragma unroll
    for (int j = 0; j < VEC; ++j) o[j] = fmaf(sc[j], g[j], fmaf(k1[j], v[j] - mu[j], k0[j]));
    storev<T, VEC>(draw + r * C + c, o);
  }
}


// ================================================================================ channel-slab kernels (clusters)
// The grid-barrier kernels above pay ~2-3 us for their barrier and a round of atomics, which is
// most of the time of the small deep-level tensors (2 - 16 MB: ~15-25 us per launch against a 1-5 us bandwidth floor).
// Here the tensor [M][C] is cut into channel SLABS of CW channels (16 or 32 bytes per row = whole sectors) and each slab
// into S row ranges: a thread-block CLUSTER of S CTAs owns one slab, every CTA reduces its rows, the S partial vectors
// are summed in rank order through distributed shared memory (one hardware cluster barrier, ~0.3 us), and each CTA
// applies the result to the rows it just read.  No global synchronisation, no workspace, bit-reproducible sums.
// Used when the slabs are short enough (levels 1-4 of a training crop); the full-resolution level (C = 32) would need
// sub-sector slabs and stays on the grid-barrier kernels.
namespace cg = cooperative_groups;
#ifndef DCB_SLAB_THREADS
#define DCB_SLAB_THREADS 512
#endif
constexpr int SLAB_THREADS = DCB_SLAB_THREADS;   // 16 warps: the dropout layers are issue bound (Philox), one CTA per SM

struct SlabGeom { int CW, S; long long rows_per_cta; };

// fixed-point thread partials (8 channels x {s, q}) -> cluster totals as doubles: lanes with the same channel group
// (lane % lanes_c) meet by shuffles, the 16 warps through shared memory, the S CTAs of the cluster through DSMEM - integer
// additions throughout, so the totals do not depend on how rows were distributed.  sh: >= 8 KB of shared memory.
__device__ __forceinline__ void slab_reduce_fixed(cg::cluster_group& cluster, long long (&s)[8], long long (&q)[8], int CW, int S,
                                                  float* sh, long long* cta_tot_q, double* s_tot, double units) {
  const int lanes_c = CW >> 3, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int off = 16; off >= lanes_c; off >>= 1) {
#pragma unroll
    for (int i = 0; i < 8; ++i) { s[i] += __shfl_xor_sync(0xffffffffu, s[i], off); q[i] += __shfl_xor_sync(0xffffffffu, q[i], off); }
  }
  long long* shq = reinterpret_cast<long long*>(sh);            // [16 warps][lanes_c <= 4][16]
  if (lane < lanes_c) {
#pragma unroll
    for (int i = 0; i < 8; ++i) { shq[(warp * 4 + lane) * 16 + i] = s[i]; shq[(warp * 4 + lane) * 16 + 8 + i] = q[i]; }
  }
  __syncthreads();
  if ((int)threadIdx.x < 2 * CW) {
    const int comp = threadIdx.x / CW, ch = threadIdx.x % CW, lc = ch >> 3, i = ch & 7;
    long long acc = 0;
    for (int w = 0; w < SLAB_THREADS / 32; ++w) acc += shq[(w * 4 + lc) * 16 + comp * 8 + i];
    cta_tot_q[threadIdx.x] = acc;
  }
  cluster.sync();
  if ((int)threadIdx.x < 2 * CW) {
    long long acc = 0;
    for (int k = 0; k < S; ++k) acc += cluster.map_shared_rank(cta_tot_q, k)[threadIdx.x];
    s_tot[threadIdx.x] = (double)acc * units;
  }
  cluster.sync();             // nobody leaves (or overwrites cta_tot_q) while a peer may still be reading it
}


template <typename T, bool POOL>
__global__ void __launch_bounds__(SLAB_THREADS)
bn_slab_fwd_kernel(const BnFwdParams p, const SlabGeom gm) {
  __shared__ __align__(16) float sh[2048];                        // 8 KB: the warps' fixed-point partials
  if (threadIdx.x == 0) pdl_trigger();
  pdl_wait();
  __shared__ double s_tot[64];
  __shared__ long long cta_tot_q[64];
  __shared__ float s_sc[32], s_sh[32];
  cg::cluster_group cluster = cg::this_cluster();
  const int C = p.C, CW = gm.CW, S = gm.S;
  const int g = blockIdx.x / S, rk = blockIdx.x % S;
  const T* __restrict__ x = reinterpret_cast<const T*>(p.x);
  const int lanes_c = CW >> 3, rows_par = SLAB_THREADS / lanes_c;
  const int tc = threadIdx.x % lanes_c, tr = threadIdx.x / lanes_c;
  const int c = g * CW + tc * 8;
  const long long r0 = (long long)rk * gm.rows_per_cta;
  long long r1 = r0 + gm.rows_per_cta; if (r1 > p.M) r1 = p.M;
  {
    FwdAcc<std::is_same<T, float>::value> sa[8], qa[8];
    long long r = r0 + tr;
    for (; r + 3LL * rows_par < r1; r += 4LL * rows_par) {
      float v[4][8];
#pragma unroll
      for (int u = 0; u < 4; ++u) load8<T>(x + (r + (long long)u * rows_par) * C + c, v[u]);
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int i = 0; i < 8; ++i) { sa[i].add(v[u][i]); qa[i].add(v[u][i] * v[u][i]); }
    }
    for (; r < r1; r += rows_par) {
      float v[8];
      load8<T>(x + r * C + c, v);
#pragma unroll
      for (int i = 0; i < 8; ++i) { sa[i].add(v[i]); qa[i].add(v[i] * v[i]); }
    }
    long long s[8], q[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { s[i] = sa[i].fixed(); q[i] = qa[i].fixed(); }
    slab_reduce_fixed(cluster, s, q, CW, S, sh, cta_tot_q, s_tot, FWD_UNITS);
  }
  __syncthreads();
  if ((int)threadIdx.x < CW) {
    const int ch = g * CW + threadIdx.x;
    const double mean = s_tot[threadIdx.x] / (double)p.M_total;
    double var = s_tot[CW + threadIdx.x] / (double)p.M_total - mean * mean;
    if (var < 0) var = 0;
    const float rstd = (float)(1.0 / sqrt(var + (double)p.eps));
    const float sc = p.gamma[ch] * rstd;
    const float shv = p.beta[ch] - (float)mean * sc;
    s_sc[threadIdx.x] = sc; s_sh[threadIdx.x] = shv;
    if (rk == 0) {
      p.scale[ch] = sc; p.shift[ch] = shv; p.mean[ch] = (float)mean; p.rstd[ch] = rstd;
      if (p.moving_mean) {   // Keras: moving <- moving*m + batch*(1-m), biased batch variance
        p.moving_mean[ch] = p.moving_mean[ch] * p.momentum + (float)mean * (1.f - p.momentum);
        p.moving_var[ch] = p.moving_var[ch] * p.momentum + (float)var * (1.f - p.momentum);
      }
    }
  }
  __syncthreads();
  float sc[8], shv[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { sc[i] = s_sc[tc * 8 + i]; shv[i] = s_sh[tc * 8 + i]; }
  unsigned long long seed = p.seed;
  if (p.seed_dev) seed ^= *p.seed_dev;
  T* __restrict__ y = reinterpret_cast<T*>(p.y);
  auto apply = [&](long long r, float (&v)[8]) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      v[j] = fmaf(v[j], sc[j], shv[j]);
      if (p.relu) v[j] = fmaxf(v[j], 0.f);
    }
    if (p.p_drop > 0.f) {
      float k[8];
      dropout_scale8(seed, p.layer, (unsigned long long)((r * C + c) >> 3), p.p_drop, k);     // same counters as the grid-barrier kernel
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] *= k[j];
    }
  };
  if constexpr (!POOL) {
    long long r = r0 + tr;
    for (; r + 3LL * rows_par < r1; r += 4LL * rows_par) {
      float v[4][8];
#pragma unroll
      for (int u = 0; u < 4; ++u) load8<T>(x + (r + (long long)u * rows_par) * C + c, v[u]);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        apply(r + (long long)u * rows_par, v[u]);
        store8<T>(y + (r + (long long)u * rows_par) * C + c, v[u]);
      }
    }
    for (; r < r1; r += rows_par) {
      float v[8];
      load8<T>(x + r * C + c, v);
      apply(r, v);
      store8<T>(y + r * C + c, v);
    }
  } else {
    // the CTA's row range is a whole number of image-row pairs (host check): pooled pixel lp of the range = rows
    // base, base+1, base+W, base+W+1 with base = r0 + (lp / OW) * 2W + 2 * (lp % OW); its flat pooled index is r0/4 + lp
    T* __restrict__ pool = reinterpret_cast<T*>(p.pool);
    const int OW = p.W >> 1;
    const long long npool = (r1 - r0) >> 2;
    auto window = [&](long long lp, float (&v)[4][8]) {
      const long long base = r0 + (lp / OW) * 2LL * p.W + 2LL * (lp % OW);
      float m[8];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const long long r = base + (k >> 1) * p.W + (k & 1);
        apply(r, v[k]);
        store8<T>(y + r * C + c, v[k]);
        // pooling compares the STORED (rounded) activations, like the standalone kernel that reads them back
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float rv = to_f32<T>(from_f32<T>(v[k][j]));
          m[j] = k == 0 ? rv : fmaxf(m[j], rv);
        }
      }
      store8<T>(pool + ((r0 >> 2) + lp) * C + c, m);
    };
    auto fetch = [&](long long lp, float (&v)[4][8]) {
      const long long base = r0 + (lp / OW) * 2LL * p.W + 2LL * (lp % OW);
#pragma unroll
      for (int k = 0; k < 4; ++k) load8<T>(x + (base + (k >> 1) * p.W + (k & 1)) * C + c, v[k]);
    };
    long long lp = tr;
    for (; lp + rows_par < npool; lp += 2LL * rows_par) {        // two windows = eight 16-byte loads in flight
      float va[4][8], vb[4][8];
      fetch(lp, va);
      fetch(lp + rows_par, vb);
      window(lp, va);
      window(lp + rows_par, vb);
    }
    for (; lp < npool; lp += rows_par) {
      float va[4][8];
      fetch(lp, va);
      window(lp, va);
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(SLAB_THREADS)
bn_slab_bwd_kernel(const BnBwdParams p, const SlabGeom gm) {
  __shared__ __align__(16) float sh[2048];                        // 8 KB: the warps' fixed-point partials
  if (threadIdx.x == 0) pdl_trigger();
  pdl_wait();
  __shared__ double s_tot[64];
  __shared__ long long cta_tot_q[64];
  cg::cluster_group cluster = cg::this_cluster();
  const int C = p.C, CW = gm.CW, S = gm.S;
  const int g = blockIdx.x / S, rk = blockIdx.x % S;
  const T* __restrict__ x = reinterpret_cast<const T*>(p.x);
  unsigned long long seed = p.seed;
  if (p.seed_dev) seed ^= *p.seed_dev;
  const int lanes_c = CW >> 3, rows_par = SLAB_THREADS / lanes_c;
  const int tc = threadIdx.x % lanes_c, tr = threadIdx.x / lanes_c;
  const int c = g * CW + tc * 8;
  const long long r0 = (long long)rk * gm.rows_per_cta;
  long long r1 = r0 + gm.rows_per_cta; if (r1 > p.M) r1 = p.M;
  float sc[8], shv[8], mu[8], rs[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { sc[i] = p.scale[c + i]; shv[i] = p.shift[c + i]; mu[i] = p.mean[c + i]; rs[i] = p.rstd[c + i]; }
  auto masked = [&](long long r, float (&gd)[8], const float (&v)[8]) {
    if (p.p_drop > 0.f) {
      float k[8];
      dropout_scale8(seed, p.layer, (unsigned long long)((r * C + c) >> 3), p.p_drop, k);
#pragma unroll
      for (int j = 0; j < 8; ++j) gd[j] *= k[j];
    }
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (fmaf(v[i], sc[i], shv[i]) <= 0.f) gd[i] = 0.f;
  };
  {
    // exact fixed-point sums (see to_q40): the same totals, bit for bit, as the grid-barrier kernel or any rank split
    BwdAcc<std::is_same<T, float>::value> sa[8], qa[8];
    long long r = r0 + tr;
    constexpr int UB = 2;                                          // rows (48 bytes of loads each) in flight per thread
    for (; r + (UB - 1LL) * rows_par < r1; r += (long long)UB * rows_par) {
      float gq[UB][8], vq[UB][8];
#pragma unroll
      for (int u = 0; u < UB; ++u) {
        load8<float>(p.dy + (r + (long long)u * rows_par) * p.ldy + p.offy + c, gq[u]);
        load8<T>(x + (r + (long long)u * rows_par) * C + c, vq[u]);
      }
#pragma unroll
      for (int u = 0; u < UB; ++u) {
        masked(r + (long long)u * rows_par, gq[u], vq[u]);
#pragma unroll
        for (int i = 0; i < 8; ++i) { sa[i].add(gq[u][i]); qa[i].add(gq[u][i] * ((vq[u][i] - mu[i]) * rs[i])); }
      }
    }
    for (; r < r1; r += rows_par) {
      float g0[8], v0[8];
      load8<float>(p.dy + r * p.ldy + p.offy + c, g0);
      load8<T>(x + r * C + c, v0);
      masked(r, g0, v0);
#pragma unroll
      for (int i = 0; i < 8; ++i) { sa[i].add(g0[i]); qa[i].add(g0[i] * ((v0[i] - mu[i]) * rs[i])); }
    }
    long long s[8], q[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { s[i] = sa[i].fixed(); q[i] = qa[i].fixed(); }
    slab_reduce_fixed(cluster, s, q, CW, S, sh, cta_tot_q, s_tot, BWD_UNITS);
  }
  __syncthreads();
  float k1[8], k0[8];
  {
    const double invM = 1.0 / (double)p.M_total;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const double scd = (double)sc[i], m1 = s_tot[tc * 8 + i] * invM, m2 = s_tot[CW + tc * 8 + i] * invM;
      k1[i] = (float)(-scd * (double)rs[i] * m2);
      k0[i] = (float)(-scd * m1);
    }
  }
  if (rk == 0 && (int)threadIdx.x < CW) {
    const int ch = g * CW + threadIdx.x;
    if (p.dbeta) p.dbeta[ch] = (float)(s_tot[threadIdx.x] * (double)p.dgb_scale);
    if (p.dgamma) p.dgamma[ch] = (float)(s_tot[CW + threadIdx.x] * (double)p.dgb_scale);
  }
  T* __restrict__ draw = reinterpret_cast<T*>(p.draw);
  long long r = r0 + tr;
  constexpr int UB = 2;
  for (; r + (UB - 1LL) * rows_par < r1; r += (long long)UB * rows_par) {
    float gq[UB][8], vq[UB][8];
#pragma unroll
    for (int u = 0; u < UB; ++u) {
      load8<float>(p.dy + (r + (long long)u * rows_par) * p.ldy + p.offy + c, gq[u]);
      load8<T>(x + (r + (long long)u * rows_par) * C + c, vq[u]);
    }
#pragma unroll
    for (int u = 0; u < UB; ++u) {
      float o[8];
      masked(r + (long long)u * rows_par, gq[u], vq[u]);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = fmaf(sc[j], gq[u][j], fmaf(k1[j], vq[u][j] - mu[j], k0[j]));
      store8<T>(draw + (r + (long long)u * rows_par) * C + c, o);
    }
  }
  for (; r < r1; r += rows_par) {
    float g0[8], v0[8], o[8];
    load8<float>(p.dy + r * p.ldy + p.offy + c, g0);
    load8<T>(x + r * C + c, v0);
    masked(r, g0, v0);
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = fmaf(sc[j], g0[j], fmaf(k1[j], v0[j] - mu[j], k0[j]));
    store8<T>(draw + r * C + c, o);
  }
}

// slab geometry for an [M][C] tensor of `esize`-byte elements; row_gran: the row ranges must be multiples of it
// (2W for the pooled forward).  false: not eligible (slabs too long, or no row split with whole ranges).
// Measured on B200 (profiles/r2_bn_slab_bench.txt): the slab kernels win where the fixed costs dominate - tensors up to
// ~4 MB forward (7.6 vs 13.4 us at 2 MB, 13.4 vs 15.6 us at 4 MB) and ~2 MB backward (8.3 vs 13.4 us) - and lose on larger
// ones, where a row-contiguous partition with four CTAs per SM streams better than one 16/32-byte column per CTA.
// policy 2 = wherever the geometry allows (tests).
static bool slab_geom(long long M, int C, int esize, long long row_gran, long long auto_max_bytes, SlabGeom& gm) {
  if (!policy(DCB_POLICY_BN_SLAB) || C % 8 != 0) return false;
  if (policy(DCB_POLICY_BN_SLAB) == 1 && M * C * esize > auto_max_bytes) return false;
  const long long max_bytes = 160 * 1024;
  for (int CW : {32 / esize, 16 / esize}) {                     // whole 32-byte sectors per row first, then half sectors
    if (CW < 8 || C % CW != 0) continue;
    const int groups = C / CW;
    for (int S = 16; S >= 1; S >>= 1) {
      if ((long long)groups * S > sm_count() + 16 && S > 1) continue;   // about one CTA per SM
      if (M % S != 0 || (M / S) % row_gran != 0) continue;
      const long long rows = M / S;
      if (rows * CW * esize > max_bytes) break;                 // a smaller S only makes the slabs longer
      if (rows < SLAB_THREADS / (CW / 8) && S > 1) continue;    // fewer rows than one pass of the CTA: split less
      gm.CW = CW; gm.S = S; gm.rows_per_cta = rows;
      return true;
    }
  }
  return false;
}

template <typename P>
static int launch_slab(void (*kernel)(P, SlabGeom), const P& p, const SlabGeom& gm, cudaStream_t st, const char* name) {
  if (int e = launch(kernel, name, (p.C / gm.CW) * gm.S, SLAB_THREADS, 0, 0, st, policy(DCB_POLICY_PDL) != 0, gm.S, p, gm)) return e;
  note_kernel(name);
  return DCB_OK;
}

// ---- host side --------------------------------------------------------------------------------------------------
static int fused_vec(int C) { return (C % 8 == 0 && 256 % (C / 8) == 0) ? 8 : ((C % 4 == 0 && 256 % (C / 4) == 0) ? 4 : 0); }

template <typename K>
static int coresident_limit(K kernel, size_t dyn_smem) {
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, dyn_smem) != cudaSuccess || per_sm < 1) return 0;
  return per_sm * sm_count();
}

static int fused_grid(long long M, int C, int vec, int limit) {
  const int rows_par = 256 / (C / vec);
  long long grid = (M + 4LL * rows_par - 1) / (4LL * rows_par);
  const int per_sm = policy(DCB_POLICY_BN_CTAS_PER_SM) > 0 ? policy(DCB_POLICY_BN_CTAS_PER_SM) : 4;
  if (grid > (long long)sm_count() * per_sm) grid = (long long)sm_count() * per_sm;
  if (grid > limit) grid = limit;
  return grid < 1 ? 1 : (int)grid;
}

static size_t fused_smem(int C, int vec) {
  const size_t phase1 = 256 * 2 * (size_t)vec * sizeof(long long);   // the backward kernel stages 64-bit partials
  const size_t phase2 = 2 * (size_t)C * sizeof(double) + 2 * (size_t)C * sizeof(float);
  return phase1 > phase2 ? phase1 : phase2;
}

static int fill_peers(PeerView& pv, const dcb_peer_exchange_t* px, int C) {
  memset(&pv, 0, sizeof(pv));
  pv.world = 1;
  if (!px || px->world <= 1) return DCB_OK;
  if (px->world > 8 || px->rank < 0 || px->rank >= px->world || !px->epoch_dev)
    return fail(DCB_ERR_INVALID_ARGUMENT, "peer exchange: bad world/rank (%d/%d) or missing epoch counter", px->world, px->rank);
  if ((long long)px->world * 2 * C > px->slot_doubles)
    return fail(DCB_ERR_INVALID_ARGUMENT, "peer exchange: slot of %lld doubles too small for %d ranks x %d values", px->slot_doubles, px->world, 2 * C);
  pv.world = px->world; pv.rank = px->rank;
  for (int i = 0; i < px->world; ++i) {
    if (!px->xchg[i] || !px->flags[i]) return fail(DCB_ERR_INVALID_ARGUMENT, "peer exchange: missing pointer for rank %d", i);
    pv.xchg[i] = reinterpret_cast<double*>(px->xchg[i]);
    pv.flags[i] = reinterpret_cast<unsigned long long*>(px->flags[i]);
  }
  pv.slot_doubles = (long long)px->slot * px->slot_doubles;
  pv.slot_flag = px->slot;
  pv.epoch = px->epoch_dev;
  return DCB_OK;
}

}  // namespace dcb

using namespace dcb;

extern "C" int dcb_bn_train_workspace_bytes(int C, size_t* bytes) {
  DCB_CHECK_ARG(bytes && C > 0, "dcb_bn_train_workspace_bytes: bad arguments");
  // the per-channel totals (64-bit fixed point)
  *bytes = 2 * (size_t)C * sizeof(long long);
  return DCB_OK;
}

#define BN_DISPATCH(dtype, ...)                                                    \
  if ((dtype) == DCB_F32) { using T = float; __VA_ARGS__ }                         \
  else if ((dtype) == DCB_BF16) { using T = __nv_bfloat16; __VA_ARGS__ }           \
  else return fail(DCB_ERR_INVALID_ARGUMENT, "training BatchNorm: dtype %d unsupported", (int)(dtype));

template <typename T, int VEC, bool POOL>
static int launch_bn_fwd(BnFwdParams& p, void* ws, size_t ws_bytes, cudaStream_t st) {
  const size_t smem = fused_smem(p.C, VEC);
  static int limit = 0;          // per template instance
  if (limit == 0) limit = coresident_limit(bn_train_fwd_kernel<T, VEC, POOL>, smem > 16384 ? smem : 16384);
  if (limit <= 0) return fail(DCB_ERR_CUDA, "occupancy query failed for the fused BatchNorm kernel");
  const int grid = fused_grid(p.M, p.C, VEC, limit);
  const size_t need = 2 * (size_t)p.C * sizeof(long long);
  if (!ws || ws_bytes < need) return fail(DCB_ERR_WORKSPACE, "dcb_bn_train_fwd: workspace %zu B < required %zu B", ws_bytes, need);
  p.totals = reinterpret_cast<double*>(ws);      // 64-bit fixed-point totals, zero on entry (see release_totals)
  if (int e = launch(bn_train_fwd_kernel<T, VEC, POOL>, "bn_train_fwd_kernel", grid, 256, smem, 0, st, policy(DCB_POLICY_PDL) != 0, 0, p))
    return e;
  note_kernel(VEC == 8 ? (POOL ? "bn_train_fwd_v8_pool" : "bn_train_fwd_v8") : (POOL ? "bn_train_fwd_v4_pool" : "bn_train_fwd_v4"));
  return DCB_OK;
}

extern "C" int dcb_bn_train_fwd(int dtype, const void* x, long long M, int C, long long M_total, const float* gamma,
                                const float* beta, float eps, float momentum, float* moving_mean, float* moving_var,
                                float* scale, float* shift, float* mean, float* rstd, int relu, float p_drop,
                                unsigned long long seed, const unsigned long long* seed_dev, unsigned layer, void* y,
                                void* pool_out, int N, int H, int W, void* workspace, size_t workspace_bytes,
                                unsigned int* sync, const dcb_peer_exchange_t* peers, dcb_stream_t stream) {
  DCB_CHECK_ARG(x && y && gamma && beta && scale && shift && mean && rstd && sync && M > 0, "dcb_bn_train_fwd: bad arguments");
  DCB_CHECK_ARG(p_drop >= 0.f && p_drop < 1.f, "dcb_bn_train_fwd: p_drop %f outside [0, 1)", p_drop);
  const int vec = fused_vec(C);
  if (!vec || C > 1024) return fail(DCB_ERR_INVALID_ARGUMENT, "dcb_bn_train_fwd: channel count %d unsupported", C);
  DCB_CHECK_ARG(!pool_out || (N > 0 && H % 2 == 0 && W % 2 == 0 && (long long)N * H * W == M), "dcb_bn_train_fwd: pooling needs N*H*W == M and even H, W");
  BnFwdParams p;
  memset(&p, 0, sizeof(p));
  p.x = x; p.y = y; p.pool = pool_out; p.M = M; p.M_total = M_total > 0 ? M_total : M; p.C = C; p.N = N; p.H = H; p.W = W;
  p.gamma = gamma; p.beta = beta; p.eps = eps; p.momentum = momentum; p.moving_mean = moving_mean; p.moving_var = moving_var;
  p.scale = scale; p.shift = shift; p.mean = mean; p.rstd = rstd; p.relu = relu; p.p_drop = p_drop; p.seed = seed;
  p.seed_dev = seed_dev; p.layer = layer; p.sync = sync;
  if (int e = fill_peers(p.pv, peers, C)) return e;
  cudaStream_t st = (cudaStream_t)stream;
  {
    SlabGeom gm;
    if (p.pv.world == 1 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0 &&
        slab_geom(M, C, dtype == DCB_F32 ? 4 : 2, pool_out ? 2LL * W : 1, 5LL << 20, gm)) {
      if (pool_out) { BN_DISPATCH(dtype, return launch_slab(bn_slab_fwd_kernel<T, true>, p, gm, st, "bn_slab_fwd_pool");) }
      else { BN_DISPATCH(dtype, return launch_slab(bn_slab_fwd_kernel<T, false>, p, gm, st, "bn_slab_fwd");) }
    }
  }
  if (vec == 8) {
    if (pool_out) { BN_DISPATCH(dtype, return (launch_bn_fwd<T, 8, true>(p, workspace, workspace_bytes, st));) }
    else { BN_DISPATCH(dtype, return (launch_bn_fwd<T, 8, false>(p, workspace, workspace_bytes, st));) }
  } else {
    if (pool_out) { BN_DISPATCH(dtype, return (launch_bn_fwd<T, 4, true>(p, workspace, workspace_bytes, st));) }
    else { BN_DISPATCH(dtype, return (launch_bn_fwd<T, 4, false>(p, workspace, workspace_bytes, st));) }
  }
}

template <typename T, int VEC, bool POOL>
static int launch_bn_fwd_sums(BnFwdParams& p, cudaStream_t st) {
  const size_t smem = fused_smem(p.C, VEC);
  // one pass, no barrier: enough CTAs to fill the machine, each with a few unrolled passes over its rows
  const int rows_par = 256 / (p.C / VEC);
  long long grid = (p.M + 8LL * rows_par - 1) / (8LL * rows_par);
  if (grid > 8LL * sm_count()) grid = 8LL * sm_count();
  if (grid < 1) grid = 1;
  if (int e = launch(bn_train_fwd_kernel<T, VEC, POOL, true>, "bn_train_fwd_kernel (sums)", (int)grid, 256, smem, 0, st,
                     policy(DCB_POLICY_PDL) != 0, 0, p))
    return e;
  note_kernel(VEC == 8 ? (POOL ? "bn_train_fwd_sums_v8_pool" : "bn_train_fwd_sums_v8")
                       : (POOL ? "bn_train_fwd_sums_v4_pool" : "bn_train_fwd_sums_v4"));
  return DCB_OK;
}

extern "C" int dcb_bn_train_fwd_sums(int dtype, const void* x, long long M, int C, long long M_total, const long long* sums_q,
                                     const float* gamma, const float* beta, float eps, float momentum, float* moving_mean,
                                     float* moving_var, float* scale, float* shift, float* mean, float* rstd, int relu,
                                     float p_drop, unsigned long long seed, const unsigned long long* seed_dev, unsigned layer,
                                     void* y, void* pool_out, int N, int H, int W, const dcb_peer_exchange_t* peers,
                                     dcb_stream_t stream) {
  DCB_CHECK_ARG(x && y && sums_q && gamma && beta && scale && shift && mean && rstd && M > 0, "dcb_bn_train_fwd_sums: bad arguments");
  DCB_CHECK_ARG(p_drop >= 0.f && p_drop < 1.f, "dcb_bn_train_fwd_sums: p_drop %f outside [0, 1)", p_drop);
  const int vec = fused_vec(C);
  if (!vec || C > 1024) return fail(DCB_ERR_INVALID_ARGUMENT, "dcb_bn_train_fwd_sums: channel count %d unsupported", C);
  DCB_CHECK_ARG(!pool_out || (N > 0 && H % 2 == 0 && W % 2 == 0 && (long long)N * H * W == M), "dcb_bn_train_fwd_sums: pooling needs N*H*W == M and even H, W");
  BnFwdParams p;
  memset(&p, 0, sizeof(p));
  p.x = x; p.y = y; p.pool = pool_out; p.M = M; p.M_total = M_total > 0 ? M_total : M; p.C = C; p.N = N; p.H = H; p.W = W;
  p.gamma = gamma; p.beta = beta; p.eps = eps; p.momentum = momentum; p.moving_mean = moving_mean; p.moving_var = moving_var;
  p.scale = scale; p.shift = shift; p.mean = mean; p.rstd = rstd; p.relu = relu; p.p_drop = p_drop; p.seed = seed;
  p.seed_dev = seed_dev; p.layer = layer; p.sums_q = sums_q;
  if (int e = fill_peers(p.pv, peers, C)) return e;
  cudaStream_t st = (cudaStream_t)stream;
  if (vec == 8) {
    if (pool_out) { BN_DISPATCH(dtype, return (launch_bn_fwd_sums<T, 8, true>(p, st));) }
    else { BN_DISPATCH(dtype, return (launch_bn_fwd_sums<T, 8, false>(p, st));) }
  } else {
    if (pool_out) { BN_DISPATCH(dtype, return (launch_bn_fwd_sums<T, 4, true>(p, st));) }
    else { BN_DISPATCH(dtype, return (launch_bn_fwd_sums<T, 4, false>(p, st));) }
  }
}

template <typename T, int VEC>
static int launch_bn_bwd(BnBwdParams& p, void* ws, size_t ws_bytes, cudaStream_t st) {
  const size_t smem = fused_smem(p.C, VEC);
  static int limit = 0;
  if (limit == 0) limit = coresident_limit(bn_train_bwd_kernel<T, VEC>, smem > 16384 ? smem : 16384);
  if (limit <= 0) return fail(DCB_ERR_CUDA, "occupancy query failed for the fused BatchNorm backward kernel");
  const int grid = fused_grid(p.M, p.C, VEC, limit);
  const size_t need = 2 * (size_t)p.C * sizeof(long long);
  if (!ws || ws_bytes < need) return fail(DCB_ERR_WORKSPACE, "dcb_bn_train_bwd: workspace %zu B < required %zu B", ws_bytes, need);
  p.totals = reinterpret_cast<double*>(ws);      // 64-bit fixed-point totals, zero on entry (see release_totals)
  if (int e = launch(bn_train_bwd_kernel<T, VEC>, "bn_train_bwd_kernel", grid, 256, smem, 0, st, policy(DCB_POLICY_PDL) != 0, 0, p))
    return e;
  note_kernel(VEC == 8 ? (p.gpix ? "bn_train_bwd_v8_rank1" : "bn_train_bwd_v8") : (p.gpix ? "bn_train_bwd_v4_rank1" : "bn_train_bwd_v4"));
  return DCB_OK;
}

static int bn_train_bwd_impl(int dtype, const float* dy, int ldy, int offy, const float* gpix, const float* wd, const void* x,
                             long long M, int C, long long M_total, const float* scale, const float* shift, const float* mean,
                             const float* rstd, float p_drop, unsigned long long seed, const unsigned long long* seed_dev,
                             unsigned layer, float dgb_scale, void* draw, float* dgamma, float* dbeta, void* workspace,
                             size_t workspace_bytes, unsigned int* sync, const dcb_peer_exchange_t* peers, dcb_stream_t stream);

extern "C" int dcb_bn_train_bwd(int dtype, const float* dy, int ldy, int offy, const void* x, long long M, int C,
                                long long M_total, const float* scale, const float* shift, const float* mean,
                                const float* rstd, float p_drop, unsigned long long seed,
                                const unsigned long long* seed_dev, unsigned layer, float dgb_scale, void* draw,
                                float* dgamma, float* dbeta, void* workspace, size_t workspace_bytes, unsigned int* sync,
                                const dcb_peer_exchange_t* peers, dcb_stream_t stream) {
  DCB_CHECK_ARG(dy, "dcb_bn_train_bwd: bad arguments");
  DCB_CHECK_ARG(ldy % 4 == 0 && offy % 4 == 0 && offy + C <= ldy, "dcb_bn_train_bwd: bad dy view (ld %d off %d C %d)", ldy, offy, C);
  DCB_CHECK_ARG((reinterpret_cast<uintptr_t>(dy) & 15) == 0, "dcb_bn_train_bwd: pointers must be 16-byte aligned");
  return bn_train_bwd_impl(dtype, dy, ldy, offy, nullptr, nullptr, x, M, C, M_total, scale, shift, mean, rstd, p_drop, seed, seed_dev,
                           layer, dgb_scale, draw, dgamma, dbeta, workspace, workspace_bytes, sync, peers, stream);
}

extern "C" int dcb_bn_train_bwd_rank1(int dtype, const float* gpix, const float* wd, const void* x, long long M, int C,
                                      long long M_total, const float* scale, const float* shift, const float* mean,
                                      const float* rstd, float p_drop, unsigned long long seed,
                                      const unsigned long long* seed_dev, unsigned layer, float dgb_scale, void* draw,
                                      float* dgamma, float* dbeta, void* workspace, size_t workspace_bytes, unsigned int* sync,
                                      const dcb_peer_exchange_t* peers, dcb_stream_t stream) {
  DCB_CHECK_ARG(gpix && wd, "dcb_bn_train_bwd_rank1: bad arguments");
  return bn_train_bwd_impl(dtype, nullptr, 0, 0, gpix, wd, x, M, C, M_total, scale, shift, mean, rstd, p_drop, seed, seed_dev, layer,
                           dgb_scale, draw, dgamma, dbeta, workspace, workspace_bytes, sync, peers, stream);
}

static int bn_train_bwd_impl(int dtype, const float* dy, int ldy, int offy, const float* gpix, const float* wd, const void* x,
                             long long M, int C, long long M_total, const float* scale, const float* shift, const float* mean,
                             const float* rstd, float p_drop, unsigned long long seed, const unsigned long long* seed_dev,
                             unsigned layer, float dgb_scale, void* draw, float* dgamma, float* dbeta, void* workspace,
                             size_t workspace_bytes, unsigned int* sync, const dcb_peer_exchange_t* peers, dcb_stream_t stream) {
  DCB_CHECK_ARG(x && scale && shift && mean && rstd && draw && sync && M > 0, "dcb_bn_train_bwd: bad arguments");
  DCB_CHECK_ARG((reinterpret_cast<uintptr_t>(x) & 15) == 0, "dcb_bn_train_bwd: pointers must be 16-byte aligned");
  const int vec = fused_vec(C);
  if (!vec || C > 1024) return fail(DCB_ERR_INVALID_ARGUMENT, "dcb_bn_train_bwd: channel count %d unsupported", C);
  BnBwdParams p;
  memset(&p, 0, sizeof(p));
  p.dy = dy; p.ldy = ldy; p.offy = offy; p.gpix = gpix; p.wd = wd; p.x = x; p.draw = draw; p.M = M; p.M_total = M_total > 0 ? M_total : M; p.C = C;
  p.scale = scale; p.shift = shift; p.mean = mean; p.rstd = rstd; p.p_drop = p_drop; p.seed = seed; p.seed_dev = seed_dev;
  p.layer = layer; p.dgb_scale = dgb_scale; p.dgamma = dgamma; p.dbeta = dbeta; p.sync = sync;
  if (int e = fill_peers(p.pv, peers, C)) return e;
  cudaStream_t st = (cudaStream_t)stream;
  {
    SlabGeom gm;
    if (!gpix && p.pv.world == 1 && (reinterpret_cast<uintptr_t>(draw) & 15) == 0 && slab_geom(M, C, dtype == DCB_F32 ? 4 : 2, 1, 5LL << 19, gm)) {
      BN_DISPATCH(dtype, return launch_slab(bn_slab_bwd_kernel<T>, p, gm, st, "bn_slab_bwd");)
    }
  }
  if (vec == 8) { BN_DISPATCH(dtype, return (launch_bn_bwd<T, 8>(p, workspace, workspace_bytes, st));) }
  else { BN_DISPATCH(dtype, return (launch_bn_bwd<T, 4>(p, workspace, workspace_bytes, st));) }
}
