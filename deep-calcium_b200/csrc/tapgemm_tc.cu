// bf16 tap-GEMM on the 5th-generation tensor cores (tcgen05.mma, fp32 accumulators in TMEM,
// operands staged in shared memory by TMA).  One persistent, warp-specialised kernel serves every
// dense contraction of the UNet2DS forward / input-gradient path (tapgeom.h):
//   conv3x3 'same' fwd + dgrad : 9 shifted [128 px x BK ch] activation boxes per K block, loaded by
//                                TMA from the NHWC tensor with out-of-bounds zero fill (= the padding)
//   convT2x2 fwd               : 1 tap, output rows scattered to (2h+a, 2w+b)
//   convT2x2 dgrad             : 4 taps read through a 5-D strided view of dy
// The channel concatenation [up | skip] (unet_2d_summary.py:200-218) is never materialised: the
// K loop walks two tensor maps.  Epilogue: acc*scale[c] + shift[c], optional ReLU, bf16 store
// (bias + BatchNorm(eps 1e-3) + ReLU folded for inference; bias only for training).
//
// CTA = 6 warps: warp 0 TMA producer, warp 1 MMA issuer (+ TMEM allocation), warps 2-5 epilogue.
// Pipelines: smem ring full/empty (TMA <-> MMA), TMEM double buffer full/empty (MMA <-> epilogue),
// static round-robin tile schedule (tile = blockIdx.x + i * gridDim.x).
#include <cstdlib>
#include <mutex>
#include <map>
#include <vector>
#include <tuple>

#include "tc_common.cuh"
#include "stats_epilogue.cuh"
#include "tapgeom.h"

namespace dcb {
using namespace tc;

constexpr int TC_BM = 128;          // pixels per tile (= UMMA M, one TMEM lane per pixel)
constexpr int TC_MAX_STAGES = 8;
constexpr int TC_THREADS = 64 + 8 * 32;   // generic kernel: TMA warp, MMA warp, two epilogue quartets (one per accumulator stage)
constexpr int ST_QUARTETS = 2;             // epilogue quartets of the strip kernel (normal orientation)
constexpr int ST_THREADS = 64 + ST_QUARTETS * 4 * 32;   // TMA warp, MMA warp, epilogue quartets
constexpr int WG_THREADS = 192;

// optional epilogue fusions requested through dcb_conv3x3_fwd_fused (mirrors dcb_conv_fusion_t)
struct TcFusion {
  const float* head_kernel; const float* head_bias; float* logit; float* prob; int need_y; void* pool_out;
};

// optional batch statistics of the output (training forward, stats_epilogue.cuh): sums[0..C) = sum, sums[C..2C) = sum of
// squares; done is set to 1 when the dispatched kernel produced them (0: the caller runs a statistics pass of its own)
struct TcStats { long long* sums; int done; };

struct TcFwdParams {
  int mode;                 // 0: 4-D halo box (conv3x3)  1: 3-D merged rows (convT fwd)  2: 5-D strided (convT dgrad)
  int N, GH, GW;            // iteration grid
  int bw, bh, bn;           // tile box in iteration-grid units (mode 1/2: bh rows of the merged N*GH axis, bn = 1)
  int tiles_w, tiles_h, tiles_n;
  int ntaps;
  int dy[9], dx[9];
  int C0, C1;               // channels of the two sources
  int BK;                   // K block (64 -> 128B swizzle, 32 -> 64B swizzle)
  int Ntot;                 // rows of the weight matrix (GEMM N over all sub-positions)
  int BN;                   // N tile (= UMMA N)
  int Cz;                   // output channels per sub-position (convT fwd: Cout, else Ntot)
  int OH, OW, OC;           // output tensor
  int osy, osx, ody, odx;   // output pixel = g * os + od (+ sub-position for convT fwd)
  int relu;
  int out_f32;              // 1: store fp32 (gradient tensors), 0: store bf16 (activations)
  int swap;                 // 1: weights are the MMA A operand (M = 128 channel rows), pixels the B operand (N = 256)
  int stages;
  int f16;                  // 16-bit element format: 0 = bf16, 1 = fp16
  int tma_store;            // 1: normal-orientation 16-bit epilogue stages blocks in smem and stores them with TMA (mapO)
  __nv_bfloat16* out;
  __nv_bfloat16* pool_out;  // conv3x3 only: 2x2 max-pooled copy [N][GH/2][GW/2][Ntot] written by the epilogue (or null)
  const float* scale;
  const float* shift;
  // STATS instantiation (training forward): per-channel sums of the stored output and of its square, see stats_epilogue.cuh
  long long* stat_sums;
};

// Epilogue of the "swapped" orientation (TMEM lane = output channel, TMEM column = pixel): each thread
// owns one channel and receives 32 consecutive pixels per tcgen05.ld; the 32 x 32 block is transposed
// through a per-warp shared-memory tile so that global stores stay NHWC-contiguous (64 B of bf16 or
// 128 B of fp32 per pixel and warp).  pix_index(m) returns the element index of pixel m's first
// channel of this warp, or -1 when the pixel lies outside the tensor.
// STATS (16-bit outputs): st_s / st_q accumulate the sum and the sum of squares of this lane's channel over the VALID pixels
// (rounded values, see stats_epilogue.cuh).
template <bool STATS = false, typename PixFn>
__device__ __forceinline__ void epilogue_swapped(uint32_t t_addr, int npix, bool warp_valid, float sc, float sh, int relu,
                                                 int out_f32, void* out_base, uint8_t* stage, int lane, PixFn pix_index,
                                                 int f16 = 0, float* st_s = nullptr, float* st_q = nullptr) {
  for (int j = 0; j < npix; j += 32) {
    uint32_t r[32];
    tmem_ld_32x32b_x32(t_addr + j, r);
    tmem_ld_wait();
    if (!warp_valid) continue;
    uint32_t vmask = 0;
    if constexpr (STATS) vmask = __ballot_sync(0xffffffffu, pix_index(j + lane) >= 0);
    __syncwarp();
    if (out_f32) {
      float* st = reinterpret_cast<float*>(stage);
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        float v = fmaf(__uint_as_float(r[i]), sc, sh);
        if (relu) v = fmaxf(v, 0.f);
        st[i * 32 + lane] = v;
      }
      __syncwarp();
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int idx = lane + 32 * q, px = idx >> 3, chunk = idx & 7;
        const long long o = pix_index(j + px);
        if (o >= 0)
          *reinterpret_cast<float4*>(reinterpret_cast<float*>(out_base) + o + chunk * 4) =
              *reinterpret_cast<const float4*>(st + px * 32 + chunk * 4);
      }
    } else {
      uint16_t* st = reinterpret_cast<uint16_t*>(stage);
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        float v = fmaf(__uint_as_float(r[i]), sc, sh);
        if (relu) v = fmaxf(v, 0.f);
        const uint16_t h = cvt16(v, f16);
        st[i * 32 + lane] = h;
        if constexpr (STATS) {
          const float rv = (vmask >> i) & 1u ? unpack16x2((uint32_t)h, f16).x : 0.f;
          *st_s += rv; *st_q = fmaf(rv, rv, *st_q);
        }
      }
      __syncwarp();
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int idx = lane + 32 * q, px = idx >> 2, chunk = idx & 3;
        const long long o = pix_index(j + px);
        if (o >= 0)
          *reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(out_base) + o + chunk * 8) =
              *reinterpret_cast<const uint4*>(st + px * 32 + chunk * 8);
      }
    }
  }
}

// Swapped orientation with the 2x2 max-pool of the encoder blocks (unet_2d_summary.py:176-194) folded in: the tile holds
// whole pairs of image rows (bw pixels wide, bw % 32 == 0), so a warp drains the 32-pixel chunk at tile position m0 (an
// even row) together with the chunk at m0 + bw (the row below), transposes both through its 4 KB shared-memory tile and
// writes the two activation rows plus the 16 pooled pixels.  16-bit outputs only.
template <typename PixFn, typename PoolFn>
__device__ __forceinline__ void epilogue_swapped_pool(uint32_t t_addr, int npix, int bw, bool warp_valid, float sc, float sh,
                                                      int relu, void* out_base, void* pool_base, uint8_t* stage, int lane,
                                                      PixFn pix_index, PoolFn pool_index, int f16) {
  uint16_t* st = reinterpret_cast<uint16_t*>(stage);            // [2 rows][32 px][32 ch]
  for (int m0 = 0; m0 < npix; m0 += 32) {
    if ((m0 / bw) & 1) continue;                                 // odd tile rows are drained with their partner
    uint32_t r0[32], r1[32];
    tmem_ld_32x32b_x32(t_addr + m0, r0);
    tmem_ld_32x32b_x32(t_addr + m0 + bw, r1);
    tmem_ld_wait();
    if (!warp_valid) continue;
    __syncwarp();
    uint16_t pooled[16];
#pragma unroll
    for (int i = 0; i < 32; i += 2) {
      float a0 = fmaf(__uint_as_float(r0[i]), sc, sh), a1 = fmaf(__uint_as_float(r0[i + 1]), sc, sh);
      float b0 = fmaf(__uint_as_float(r1[i]), sc, sh), b1 = fmaf(__uint_as_float(r1[i + 1]), sc, sh);
      if (relu) { a0 = fmaxf(a0, 0.f); a1 = fmaxf(a1, 0.f); b0 = fmaxf(b0, 0.f); b1 = fmaxf(b1, 0.f); }
      st[i * 32 + lane] = cvt16(a0, f16);
      st[(i + 1) * 32 + lane] = cvt16(a1, f16);
      st[1024 + i * 32 + lane] = cvt16(b0, f16);
      st[1024 + (i + 1) * 32 + lane] = cvt16(b1, f16);
      // rounding is monotonic: the maximum of the rounded values is the rounded maximum
      pooled[i >> 1] = cvt16(fmaxf(fmaxf(a0, a1), fmaxf(b0, b1)), f16);
    }
    __syncwarp();
#pragma unroll
    for (int q = 0; q < 8; ++q) {                                // 2 rows x 32 px x 4 chunks of 8 channels
      const int idx = lane + 32 * q, row = idx >> 7, px = (idx >> 2) & 31, chunk = idx & 3;
      const long long o = pix_index(m0 + row * bw + px);
      if (o >= 0)
        *reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(out_base) + o + chunk * 8) =
            *reinterpret_cast<const uint4*>(st + row * 1024 + px * 32 + chunk * 8);
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 16; ++k) st[k * 32 + lane] = pooled[k];
    __syncwarp();
#pragma unroll
    for (int q = 0; q < 2; ++q) {                                // 16 pooled px x 4 chunks
      const int idx = lane + 32 * q, pp = idx >> 2, chunk = idx & 3;
      const long long o = pool_index(m0 + 2 * pp);
      if (o >= 0)
        *reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(pool_base) + o + chunk * 8) =
            *reinterpret_cast<const uint4*>(st + pp * 32 + chunk * 8);
    }
    __syncwarp();
  }
}

// POOL: the epilogues also write the 2x2 max-pooled copy (p.pool_out); a separate instantiation so that the plain
// kernel keeps its register allocation (the pooled epilogue cost the plain path ~10 % when it was a runtime branch)
// STATS: normal orientation, 16-bit plain stores; the epilogue also accumulates the BatchNorm batch statistics
template <bool POOL, bool STATS>
__global__ void __launch_bounds__(TC_THREADS, 1)
tapgemm_tc_fwd_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
                      const __grid_constant__ CUtensorMap mapB, const __grid_constant__ CUtensorMap mapO, const TcFwdParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ uint64_t bar_full[TC_MAX_STAGES], bar_empty[TC_MAX_STAGES], bar_tfull[2], bar_tempty[2];
  __shared__ uint32_t tmem_base_smem;
  __shared__ __align__(16) float s_scale[512], s_shift[512];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) pdl_trigger();
  // dynamic smem: 1024-byte aligned stage buffers (swizzle atoms are address based)
  // 1024-byte alignment as an offset into the __shared__ array (an integer round trip would turn every later access
  // through this pointer into a generic-space load/store)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  // pixel tile: 128 rows (normal) or 256 rows (swapped); weight tile: BN rows (normal) or 128 rows (swapped)
  const int PX = p.swap ? 256 : TC_BM;
  const uint32_t a_bytes = PX * p.BK * 2, b_bytes = (p.swap ? 128 : p.BN) * p.BK * 2;
  const uint32_t stage_bytes = a_bytes + b_bytes;
  const int kb0 = p.C0 / p.BK, kb1 = p.C1 / p.BK;
  const int kb_per_tap = kb0 + kb1;
  const int num_kb = p.ntaps * kb_per_tap;
  const int Ktap = p.C0 + p.C1;
  const int num_ntiles = p.swap ? (p.Ntot + 127) / 128 : p.Ntot / p.BN;
  const int num_mtiles = p.tiles_w * p.tiles_h * p.tiles_n;
  const int num_tiles = num_mtiles * num_ntiles;
  const int acc_cols = p.swap ? 256 : p.BN;          // TMEM columns per accumulator stage
  uint32_t tmem_cols = 32;
  while (tmem_cols < 2u * acc_cols) tmem_cols <<= 1;
  __shared__ __align__(16) uint8_t s_stage[4][4096];  // per-epilogue-warp transpose tiles (swapped mode; STATS: 8 x 2 KB)
  // STATS: this lane's sums of channel pair (lane & 15) of accumulator block bi, over all tiles of the CTA
  float2 st_s[STATS ? 8 : 1], st_q[STATS ? 8 : 1];
#pragma unroll
  for (int i = 0; i < (STATS ? 8 : 1); ++i) { st_s[i] = make_float2(0.f, 0.f); st_q[i] = make_float2(0.f, 0.f); }

  for (int i = threadIdx.x; i < p.Cz; i += blockDim.x) {
    s_scale[i] = p.scale ? p.scale[i] : 1.f;
    s_shift[i] = p.shift ? p.shift[i] : 0.f;
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapA0);
    if (p.C1 > 0) tma_prefetch_desc(&mapA1);
    tma_prefetch_desc(&mapB);
    for (int s = 0; s < p.stages; ++s) { mbar_init(&bar_full[s], 1); mbar_init(&bar_empty[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&bar_tfull[s], 1); mbar_init(&bar_tempty[s], 4); }
    mbar_fence_init();
  }
  if (warp == 1) {
    tmem_alloc(&tmem_base_smem, tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;

  if (warp == 0) {
    // ===================================================== TMA producer
    if (elect_one()) {
      int stage = 0; uint32_t phase = 0;
      pdl_wait();                                   // the activations come from the previous kernel of the stream
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int nt = tile % num_ntiles, mt = tile / num_ntiles;
        const int tw = mt % p.tiles_w, th = (mt / p.tiles_w) % p.tiles_h, tn = mt / (p.tiles_w * p.tiles_h);
        const int w0 = tw * p.bw, h0 = th * p.bh, n0 = tn * p.bn;
        for (int tap = 0; tap < p.ntaps; ++tap) {
          for (int kk = 0; kk < kb_per_tap; ++kk) {
            const bool second = kk >= kb0;
            const int c0 = (second ? kk - kb0 : kk) * p.BK;
            const CUtensorMap* mA = second ? &mapA1 : &mapA0;
            mbar_wait(&bar_empty[stage], phase ^ 1);
            uint8_t* sa = smem + (size_t)stage * stage_bytes;
            uint8_t* sb = sa + a_bytes;
            // swapped: the weight box holds min(128, rows left) rows; the rest of the 128-row A tile is stale
            // shared memory that only feeds accumulator lanes nobody reads
            const int wrows = p.swap ? (p.Ntot - nt * 128 < 128 ? p.Ntot - nt * 128 : 128) : p.BN;
            mbar_arrive_expect_tx(&bar_full[stage], a_bytes + (uint32_t)wrows * p.BK * 2);
            if (p.mode == 0) tma_load_4d(mA, &bar_full[stage], sa, c0, w0 + p.dx[tap], h0 + p.dy[tap], n0);
            else if (p.mode == 1) tma_load_3d(mA, &bar_full[stage], sa, c0, w0, h0);
            else tma_load_5d(mA, &bar_full[stage], sa, c0, p.dx[tap], w0, p.dy[tap], h0);
            tma_load_2d(&mapB, &bar_full[stage], sb, tap * Ktap + (second ? p.C0 : 0) + c0, nt * (p.swap ? 128 : p.BN));
            if (++stage == p.stages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================================================== MMA issuer (single thread)
    if (elect_one()) {
      const uint32_t idesc = p.swap ? make_idesc_16(128, 256, 0, 0, p.f16) : make_idesc_16(TC_BM, p.BN, 0, 0, p.f16);
      const uint32_t swz = (p.BK == 64) ? SWZ_128B : SWZ_64B;
      const uint32_t sbo = 8u * p.BK * 2u;          // 8 rows of BK bf16
      const int ksteps = p.BK / 16;
      const uint64_t dbase = make_smem_desc(0, 16, sbo, swz);
      const uint32_t smem16 = smem_u32(smem) >> 4, stage16 = stage_bytes >> 4, a16 = a_bytes >> 4;
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      // Split-phase polling of the stage barriers (see the folded strip loop): the non-blocking test of the NEXT
      // stage's full barrier is issued before this stage's MMAs and consumed one iteration later, so its ~250 cycles
      // of latency overlap with the MMA issue instead of adding to the 4 x 128 cycles a stage keeps the pipe busy.
      const uint32_t a_full = smem_u32_pinned(bar_full), a_empty = smem_u32_pinned(bar_empty);
      asm volatile(".reg .pred p_full;");
      bool pre = false;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        mbar_wait(&bar_tempty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * acc_cols);
        for (int kb = 0; kb < num_kb; ++kb) {
          {
            uint32_t ok = 0;
            if (pre) asm volatile("selp.u32 %0, 1, 0, p_full;" : "=r"(ok));
            if (!ok) mbar_wait_a(a_full + 8u * stage, phase);
            int ns = stage + 1; uint32_t np = phase;
            if (ns == p.stages) { ns = 0; np ^= 1u; }
            asm volatile("mbarrier.test_wait.parity.shared::cta.b64 p_full, [%0], %1;" ::"r"(a_full + 8u * ns), "r"(np) : "memory");
            pre = true;
          }
          tc_fence_after();
          // descriptors differ only in the 14-bit start-address field: one add per operand and K step keeps
          // the single issuing thread far below the ~89-128 cycles an MMA occupies the tensor pipe
          const uint32_t sa16 = smem16 + (uint32_t)stage * stage16, sb16 = sa16 + a16;
          const uint64_t da = dbase + (p.swap ? sb16 : sa16);   // swapped: A = weight tile, B = pixel tile
          const uint64_t db = dbase + (p.swap ? sa16 : sb16);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            // advance 16 bf16 = 32 bytes along K inside the swizzle atom: +2 in the (addr >> 4) field
            if (k < ksteps) umma_bf16(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
          }
          umma_commit_a(a_empty + 8u * stage);       // smem slot free once these MMAs retire
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&bar_tfull[acc]);                // accumulator ready for the epilogue
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    // ===================================================== epilogue warps (TMEM -> regs -> global)
    const int quarter = warp & 3;                    // TMEM lanes [32*quarter, 32*quarter+32)
    const int m = quarter * 32 + lane;               // row of the tile = pixel
    // Normal orientation: two quartets, quartet q drains accumulator stage q (every other tile) - draining a
    // [128 x BN] accumulator takes one quartet longer than the MMAs of a short-K tile (convT: K = Cin only).
    // Swapped orientation: one quartet (its transpose buffers are per warp), the second one idles.
    const int eset = (warp - 2) >> 2, nsets = p.swap ? 1 : 2;
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < num_tiles && eset < nsets; tile += gridDim.x, ++it) {
      if (nsets == 2 && (int)(it & 1u) != eset) continue;
      const int acc = (int)(it & 1u);
      const uint32_t acc_phase = (it >> 1) & 1u;
      const int nt = tile % num_ntiles, mt = tile / num_ntiles;
      const int tw = mt % p.tiles_w, th = (mt / p.tiles_w) % p.tiles_h, tn = mt / (p.tiles_w * p.tiles_h);
      if (p.swap) {
        // lane = GEMM row (output channel incl. convT sub-position), column = pixel of the 256-pixel tile
        const int grow = nt * 128 + quarter * 32;          // first GEMM row of this warp
        const bool warp_valid = grow < p.Ntot;
        const int z = grow / p.Cz, cw = grow % p.Cz;
        const int ody = p.Cz < p.Ntot ? (z >> 1) : p.ody, odx = p.Cz < p.Ntot ? (z & 1) : p.odx;
        const float sc = warp_valid ? s_scale[cw + lane] : 0.f, sh = warp_valid ? s_shift[cw + lane] : 0.f;
        auto pix_index = [&](int mm) -> long long {
          int n2, gh2, gw2;
          if (p.mode == 0) {
            gw2 = tw * p.bw + mm % p.bw;
            gh2 = th * p.bh + (mm / p.bw) % p.bh;
            n2 = tn * p.bn + mm / (p.bw * p.bh);
            if (gw2 >= p.GW || gh2 >= p.GH || n2 >= p.N) return -1;
          } else {
            gw2 = tw * p.bw + mm % p.bw;
            const int r2 = th * p.bh + mm / p.bw;
            if (gw2 >= p.GW || r2 >= p.N * p.GH) return -1;
            n2 = r2 / p.GH; gh2 = r2 % p.GH;
          }
          return (long long)((((size_t)n2 * p.OH + (gh2 * p.osy + ody)) * p.OW + (gw2 * p.osx + odx)) * p.OC + cw);
        };
        mbar_wait(&bar_tfull[acc], acc_phase);
        tc_fence_after();
        if constexpr (POOL) {
          // pooled index of tile position mm (even row, even column of the tile; the host guarantees even GH, GW, bw, bh)
          auto pool_index = [&](int mm) -> long long {
            const int gw2 = tw * p.bw + mm % p.bw, gh2 = th * p.bh + (mm / p.bw) % p.bh, n2 = tn * p.bn + mm / (p.bw * p.bh);
            if (gw2 >= p.GW || gh2 >= p.GH || n2 >= p.N) return -1;
            return (long long)((((size_t)n2 * (p.GH >> 1) + (gh2 >> 1)) * (p.GW >> 1) + (gw2 >> 1)) * p.OC + cw);
          };
          epilogue_swapped_pool(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * acc_cols), 256, p.bw, warp_valid, sc,
                                sh, p.relu, p.out, p.pool_out, s_stage[quarter], lane, pix_index, pool_index, p.f16);
        } else {
          epilogue_swapped(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * acc_cols), 256, warp_valid, sc, sh,
                           p.relu, p.out_f32, p.out, s_stage[quarter], lane, pix_index, p.f16);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_tempty[acc]);
        continue;
      }
      // pixel of this row
      int n, gh, gw;
      bool valid;
      if (p.mode == 0) {
        gw = tw * p.bw + m % p.bw;
        gh = th * p.bh + (m / p.bw) % p.bh;
        n = tn * p.bn + m / (p.bw * p.bh);
        valid = gw < p.GW && gh < p.GH && n < p.N;
      } else {
        gw = tw * p.bw + m % p.bw;
        const int r = th * p.bh + m / p.bw;
        n = r / p.GH; gh = r % p.GH;
        valid = gw < p.GW && r < p.N * p.GH;
      }
      const int ng0 = nt * p.BN;                     // first GEMM column of this tile
      // pixel part of the output index; the sub-position (convT fwd) depends on the 32-column block
      const size_t orow_y = (size_t)n * p.OH + gh * p.osy;
      const int ocol_x = gw * p.osx;

      mbar_wait(&bar_tfull[acc], acc_phase);
      tc_fence_after();
      const uint32_t t_addr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * p.BN);
      if constexpr (STATS) {
        // one 32-column block at a time: pack, store, and feed the packed block to the statistics (the shared-memory
        // transpose of stats_block is the second instruction stream here)
        int z = ng0 / p.Cz, ch = ng0 - z * p.Cz;
        const bool subpos = p.Cz < p.Ntot;
        uint32_t* scr = reinterpret_cast<uint32_t*>(&s_stage[0][0]) + (warp - 2) * STATS_SCRATCH_WORDS;
#pragma unroll
        for (int bi = 0; bi < 8; ++bi) {
          if (bi * 32 < p.BN) {
            uint32_t r[32];
            tmem_ld_32x32b_x32(t_addr + bi * 32, r);
            tmem_ld_wait();
            uint32_t pk[16];
            bn_relu_pack32(r, s_scale + ch, s_shift + ch, p.relu, pk, p.f16);
            if (valid) {
              const int ody = subpos ? (z >> 1) : p.ody, odx = subpos ? (z & 1) : p.odx;
              store_pk16(p.out + ((orow_y + ody) * p.OW + (ocol_x + odx)) * p.OC + ch, pk);
            }
            stats_block(pk, valid, scr, lane, p.f16, st_s[bi], st_q[bi]);
            ch += 32; if (ch == p.Cz) { ch = 0; ++z; }
          }
        }
      } else if constexpr (!POOL) {
        // Two 32-column blocks per step: their TMEM loads, BN / ReLU / pack arithmetic and stores are independent
        // instruction streams (each scheduler hosts two epilogue warps, so a block-at-a-time loop is latency bound -
        // the short-K convT tiles spend 3x longer in this epilogue than in their MMAs).  A block never straddles a
        // convT sub-position because Cz % 32 == 0; (z, ch) = sub-position and channel of a block, advanced without divisions.
        int z = ng0 / p.Cz, ch = ng0 - z * p.Cz;
        const bool subpos = p.Cz < p.Ntot;
        auto out_index = [&](int zz, int cc) -> size_t {
          const int ody = subpos ? (zz >> 1) : p.ody, odx = subpos ? (zz & 1) : p.odx;
          return ((orow_y + ody) * p.OW + (ocol_x + odx)) * p.OC + cc;
        };
        auto store_f32 = [&](const uint32_t (&r)[32], int cc, size_t o) {
          float* orow_f = reinterpret_cast<float*>(p.out) + o;
#pragma unroll
          for (int q0 = 0; q0 < 32; q0 += 8) {
            uint32_t v[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              float f = fmaf(__uint_as_float(r[q0 + q]), s_scale[cc + q0 + q], s_shift[cc + q0 + q]);
              if (p.relu) f = fmaxf(f, 0.f);
              v[q] = __float_as_uint(f);
            }
            st_global_v8(orow_f + q0, v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7]);
          }
        };
        // TMA-store mode: per quartet two 8 KB staging tiles ([128 px][32 ch], SWIZZLE_64B) behind the stage ring
        const uint32_t stg = smem_u32(smem + (size_t)p.stages * stage_bytes) + (uint32_t)eset * 16384u;
        const bool leader = quarter == 0 && lane == 0;
        for (int c = 0; c < p.BN; c += 64) {
          const bool two = c + 32 < p.BN;
          const int z0 = z, ch0 = ch;
          ch += 32; if (ch == p.Cz) { ch = 0; ++z; }
          const int z1 = z, ch1 = ch;
          if (two) { ch += 32; if (ch == p.Cz) { ch = 0; ++z; } }
          uint32_t r0[32], r1[32];
          tmem_ld_32x32b_x32(t_addr + c, r0);
          if (two) tmem_ld_32x32b_x32(t_addr + c + 32, r1);
          tmem_ld_wait();
          if (p.tma_store) {
            uint32_t pk0[16], pk1[16];
            bn_relu_pack32(r0, s_scale + ch0, s_shift + ch0, p.relu, pk0, p.f16);
            if (two) bn_relu_pack32(r1, s_scale + ch1, s_shift + ch1, p.relu, pk1, p.f16);
            if (leader) bulk_wait_read0();                       // the previous stores have read the staging tiles
            named_bar_sync(1 + eset, 128);
            stage_pk16_swz64(stg, m, pk0);
            if (two) stage_pk16_swz64(stg + 8192u, m, pk1);
            fence_proxy_async_smem();
            named_bar_sync(1 + eset, 128);
            if (leader) {
              const int w0 = tw * p.bw, h0 = th * p.bh;
              if (p.mode == 0) {
                tma_store_4d(&mapO, smem + (size_t)p.stages * stage_bytes + eset * 16384, ch0, w0, h0, tn * p.bn);
                if (two) tma_store_4d(&mapO, smem + (size_t)p.stages * stage_bytes + eset * 16384 + 8192, ch1, w0, h0, tn * p.bn);
              } else {
                tma_store_5d(&mapO, smem + (size_t)p.stages * stage_bytes + eset * 16384, ch0, z0 & 1, w0, z0 >> 1, h0);
                if (two) tma_store_5d(&mapO, smem + (size_t)p.stages * stage_bytes + eset * 16384 + 8192, ch1, z1 & 1, w0, z1 >> 1, h0);
              }
              bulk_commit();
            }
            continue;
          }
          const size_t o0 = out_index(z0, ch0), o1 = out_index(z1, ch1);
          if (!valid) continue;
          if (p.out_f32) {
            store_f32(r0, ch0, o0);
            if (two) store_f32(r1, ch1, o1);
          } else if (two) {
            uint32_t pk0[16], pk1[16];
            bn_relu_pack32(r0, s_scale + ch0, s_shift + ch0, p.relu, pk0, p.f16);
            bn_relu_pack32(r1, s_scale + ch1, s_shift + ch1, p.relu, pk1, p.f16);
            store_pk16(p.out + o0, pk0);
            store_pk16(p.out + o1, pk1);
          } else {
            uint32_t pk0[16];
            bn_relu_pack32(r0, s_scale + ch0, s_shift + ch0, p.relu, pk0, p.f16);
            store_pk16(p.out + o0, pk0);
          }
        }
      } else
      for (int c = 0; c < p.BN; c += 32) {
        // a 32-column block never straddles a sub-position because Cz % 32 == 0
        const int gcol = ng0 + c;
        const int z = gcol / p.Cz, cbase = gcol % p.Cz - c;   // cbase + c = channel of the block's first column
        const int ody = p.Cz < p.Ntot ? (z >> 1) : p.ody, odx = p.Cz < p.Ntot ? (z & 1) : p.odx;
        const size_t oidx = ((orow_y + ody) * p.OW + (ocol_x + odx)) * p.OC + cbase;
        __nv_bfloat16* orow = p.out + oidx;
        float* orow_f = reinterpret_cast<float*>(p.out) + oidx;
        uint32_t r[32];
        tmem_ld_32x32b_x32(t_addr + c, r);
        tmem_ld_wait();
        if (valid && p.out_f32) {
#pragma unroll
          for (int j = 0; j < 32; j += 8) {
            uint32_t v[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const int ch = cbase + c + j + q;
              float f = fmaf(__uint_as_float(r[j + q]), s_scale[ch], s_shift[ch]);
              if (p.relu) f = fmaxf(f, 0.f);
              v[q] = __float_as_uint(f);
            }
            st_global_v8(orow_f + c + j, v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7]);
          }
        } else if (valid || POOL) {
          uint32_t pk[16];
          bn_relu_pack32(r, s_scale + cbase + c, s_shift + cbase + c, p.relu, pk, p.f16);
          if (valid) store_pk16(orow + c, pk);
          if constexpr (POOL) {
            // 2x2 max-pool folded in (unet_2d_summary.py:176-194): the tile holds whole 2x2 windows (even bw, bh and even
            // image sizes, checked on the host).  The quartet exchanges the packed 32-channel blocks through its 8 KB of
            // the (otherwise unused) transpose buffer; named barrier 1 + eset = the 128 threads of this quartet.
            uint4* stg = reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(s_stage) + eset * 8192);
#pragma unroll
            for (int q = 0; q < 4; ++q) stg[m * 4 + q] = make_uint4(pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
            asm volatile("bar.sync %0, 128;" ::"r"(1 + eset) : "memory");
            const int lx = m % p.bw, ly = (m / p.bw) % p.bh;
            if (valid && !(lx & 1) && !(ly & 1)) {
              uint32_t mx[16];
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const uint4 b4 = stg[(m + 1) * 4 + q], c4 = stg[(m + p.bw) * 4 + q], d4 = stg[(m + p.bw + 1) * 4 + q];
                mx[4 * q] = max16x2(max16x2(pk[4 * q], b4.x, p.f16), max16x2(c4.x, d4.x, p.f16), p.f16);
                mx[4 * q + 1] = max16x2(max16x2(pk[4 * q + 1], b4.y, p.f16), max16x2(c4.y, d4.y, p.f16), p.f16);
                mx[4 * q + 2] = max16x2(max16x2(pk[4 * q + 2], b4.z, p.f16), max16x2(c4.z, d4.z, p.f16), p.f16);
                mx[4 * q + 3] = max16x2(max16x2(pk[4 * q + 3], b4.w, p.f16), max16x2(c4.w, d4.w, p.f16), p.f16);
              }
              store_pk16(p.pool_out + (((size_t)n * (p.GH >> 1) + (gh >> 1)) * (p.GW >> 1) + (gw >> 1)) * p.OC + cbase + c, mx);
            }
            asm volatile("bar.sync %0, 128;" ::"r"(1 + eset) : "memory");
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_tempty[acc]);
    }
    if (p.tma_store && quarter == 0 && lane == 0) bulk_wait0();   // staging tiles stay valid until the last store is done
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
  if constexpr (STATS) {
    // every MMA has retired: the stage ring is free and takes the per-warp accumulators ([8 warps][nblk][16][4] floats)
    float* dump = reinterpret_cast<float*>(smem);
    const int nblk = p.BN / 32;
    if (warp >= 2 && lane < 16) {
#pragma unroll
      for (int bi = 0; bi < 8; ++bi)
        if (bi < nblk)
          *reinterpret_cast<float4*>(dump + ((size_t)((warp - 2) * nblk + bi) * 16 + lane) * 4) =
              make_float4(st_s[bi].x, st_s[bi].y, st_q[bi].x, st_q[bi].y);
    }
    __syncthreads();
    // the host launches a multiple of num_ntiles CTAs, so every tile of this CTA has the same N tile
    const int nt = blockIdx.x % num_ntiles;
    stats_cta_finish(dump, 8, nblk, [&](int bi) { return (nt * p.BN + bi * 32) % p.Cz; }, p.Cz, p.stat_sums);
  }
}

// ====================================================================================== strip kernel
// conv3x3 for the wide, shallow layers (W % 128 == 0, 9*Cin*Cout*2 bytes of weights fit in smem):
// the layers where the generic kernel is bound by re-loading the activations 9x (once per tap).
//   * all 9 x nkc weight tiles stay resident in shared memory for the whole (persistent) CTA;
//   * a CTA walks a strip of output rows x 128 pixels (balanced partition, see the kernel); the producer streams
//     the strip's rows + 2 halo rows ([130 px x BK ch] TMA boxes, zero filled outside the image) through a ring,
//     so every activation row is fetched about once instead of 9 times;
//   * the three horizontal taps read the SAME halo row: the A descriptor simply starts dx pixels
//     (dx * row pitch bytes) further into the swizzled tile.  The swizzle XOR is a function of the
//     absolute smem address, so a row-shifted start address needs no base-offset correction
//     (verified on B200: profiles/r1_umma_row_shift_probe.log);
//   * the three vertical taps read three consecutive ring rows (plain mode) or are folded into the MMA N
//     dimension (FOLD mode, see the kernel).
// Plain-mode MMA issue of one strip tile: 9 taps x nkc channel chunks x KSTEPS MMAs.  Templated so that the single issuing
// thread runs straight-line code (every extra dependent instruction between two tcgen05.mma shows up directly
// in the tensor-pipe utilisation of these short-K tiles).  Weight tiles are laid out (tap, kc)-major, so the
// weight descriptor simply advances by one tile per step.
template <int KSTEPS, bool SWAP>
__device__ __forceinline__ void strip_issue_tile(uint32_t d_tmem, uint64_t dbase, const uint32_t (&row16)[3], uint32_t w16,
                                                 int nkc, uint32_t slot16, uint32_t pitch16, uint32_t wblk16, uint32_t idesc) {
  // Order: consecutive MMAs read DIFFERENT halo rows (dy innermost).  Back-to-back MMAs whose A operands are the
  // same rows shifted by one pixel issue ~2x slower (measured, profiles/r1_strip_scaling.txt).
  const uint32_t wtap16 = (uint32_t)nkc * wblk16;
  uint32_t accf = 0;
  for (int kc = 0; kc < nkc; ++kc) {
#pragma unroll
    for (int dx = 0; dx < 3; ++dx) {
#pragma unroll
      for (int k = 0; k < KSTEPS; ++k) {
#pragma unroll
        for (int dy = 0; dy < 3; ++dy) {
          const uint64_t dpx = dbase + (row16[dy] + kc * slot16 + dx * pitch16 + 2 * k);
          const uint64_t dwt = dbase + (w16 + (dy * 3 + dx) * wtap16 + kc * wblk16 + 2 * k);
          if (SWAP) umma_bf16(d_tmem, dwt, dpx, idesc, accf);
          else umma_bf16(d_tmem, dpx, dwt, idesc, accf);
          accf = 1;
        }
      }
    }
  }
}

// Folded mode (see the strip kernel): all steps of one halo row except the first; each step is one MMA (or two when
// the accumulator ring wraps inside the span).  Weight groups are (kc, dx)-major: three stacked tiles per group.
template <int KSTEPS, bool TWO>
__device__ __forceinline__ void fold_issue_rest(uint32_t d0, uint32_t d1, uint64_t dA, uint64_t dW0, uint64_t dW1, uint32_t idesc0,
                                                uint32_t idesc1, int nkc, uint32_t slot16, uint32_t pitch16, uint32_t wblk16) {
  for (int kc = 0; kc < nkc; ++kc) {
#pragma unroll
    for (int dx = 0; dx < 3; ++dx) {
#pragma unroll
      for (int k = 0; k < KSTEPS; ++k) {
        if (kc == 0 && dx == 0 && k == 0) continue;
        const uint32_t ao = kc * slot16 + dx * pitch16 + 2 * k, wo = (uint32_t)(kc * 3 + dx) * 3u * wblk16 + 2 * k;
        umma_bf16(d0, dA + ao, dW0 + wo, idesc0, 1u);
        if (TWO) umma_bf16(d1, dA + ao, dW1 + wo, idesc1, 1u);
      }
    }
  }
}

// Folded mode, interior halo row whose three accumulators do not wrap around the ring: the weight descriptors are
// loop invariant, only the row descriptor dA and the accumulator address d0 change.  First step: rows i-1, i
// accumulate (N = 2*Cout), row i+1 is opened with accumulate = 0 (N = Cout); then N = 3*Cout.
template <int KSTEPS>
__device__ __forceinline__ void fold_issue_fast(uint32_t d0, uint32_t d2, uint64_t dA, uint64_t dW, uint32_t id1, uint32_t id2,
                                                uint32_t id3, int nkc, uint32_t slot16, uint32_t pitch16, uint32_t wblk16) {
  umma_bf16(d0, dA, dW, id2, 1u);
  umma_bf16(d2, dA, dW + 2u * wblk16, id1, 0u);
  for (int kc = 0; kc < nkc; ++kc) {
#pragma unroll
    for (int dx = 0; dx < 3; ++dx) {
#pragma unroll
      for (int k = 0; k < KSTEPS; ++k) {
        if (kc == 0 && dx == 0 && k == 0) continue;
        umma_bf16(d0, dA + (kc * slot16 + dx * pitch16 + 2 * k), dW + ((uint32_t)(kc * 3 + dx) * 3u * wblk16 + 2 * k), id3, 1u);
      }
    }
  }
}

constexpr int ST_MAX_RING = 12;

// ---- thread-block cluster helpers (CTA-pair kernels below)
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// bulk-tensor load delivered to the same shared-memory offset of every CTA in ctaMask; each destination CTA's mbarrier (same
// offset) receives the complete_tx
__device__ __forceinline__ void tma_load_4d_mc(const CUtensorMap* m, uint64_t* bar, void* dst, int c0, int c1, int c2, int c3,
                                               uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4, %5, %6}], [%2], %7;"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "h"(cta_mask)
      : "memory");
}
// single-CTA MMAs, completion signalled on the barrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_mc2(uint32_t bar_addr) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar_addr), "h"((uint16_t)3) : "memory");
}

// -DDCB_STRIP_TIMING: the folded MMA thread accumulates clock64() intervals (diagnostic builds only)
#ifdef DCB_STRIP_TIMING
__device__ unsigned long long g_strip_dbg[148 * 8];
__device__ unsigned long long g_strip_dbg2[148 * 16];
#define ST_T(var) const long long var = clock64()
#define ST_DECL(var) long long var = 0
#define ST_SET(var) var = clock64()
#define ST_ACC(slot, a, b) dbg_acc[slot] += (unsigned long long)((b) - (a))
#else
#define ST_T(var)
#define ST_DECL(var)
#define ST_SET(var)
#define ST_ACC(slot, a, b)
#endif

struct TcStripParams {
  int N, H, W;
  int C0, C1, BK, nkc;
  int Cout;
  int ring, wsegs;
  int gran;                 // partition granularity in rows (2 when H is even: fused pool pairs stay inside a strip)
  int slot_bytes;           // (PX + 2) * BK * 2 rounded up to 1024
  int swap;                 // 1: 256-pixel segments, weights as the MMA A operand (see TcFwdParams::swap)
  int fold;                 // 1: the three vertical taps are folded into the MMA N dimension (see the kernel comment)
  int OC, n0;               // output tensor channel pitch and first output channel of this launch (Cout = channels computed here)
  int nclu;                 // 2: clusters of two CTAs compute the two Cout-channel halves of the SAME pixels (folded mode): CTA r
                            // takes channels n0 + r*Cout.., each halo row is fetched once and TMA-multicast into both CTAs
                            // (the two channel-split launches of a 128 -> 64 layer each read the whole input)
  // optional epilogue fusions (normal orientation only)
  const float* head_kernel; // [Cout][2] softmax head (unet_2d_summary.py:221-222): emit logit / prob per pixel
  const float* head_bias;   // [2]
  float* logit; float* prob;
  int need_y;               // 0: the activation itself is not stored (head fused, nobody else reads it)
  __nv_bfloat16* pool_out;  // 2x2 max-pooled copy [N][H/2][W/2][Cout] (unet_2d_summary.py:176-194) or null
  int relu, out_f32;
  int f16;                  // 16-bit element format: 0 = bf16, 1 = fp16
  __nv_bfloat16* out;
  const float* scale;
  const float* shift;
  // STATS instantiation (training forward): per-channel sums of the stored output and of its square, see stats_epilogue.cuh
  long long* stat_sums;
};

// per-lane statistics accumulators of the strip epilogue (Cout <= 64: two 32-channel blocks) + the warp's scratch tile
struct StripStats { float2 s[2], q[2]; uint32_t* scr; };

// Drains one PAIR of output rows of a folded strip (accumulators at TMEM addresses ta / tb, lane = pixel): BN / ReLU / pack,
// optional fused softmax head and 2x2 max-pool, 16-bit or fp32 stores.  Both rows are processed together: the two TMEM
// loads, the arithmetic and the stores of the two rows are independent instruction streams (twice the ILP of a
// row-at-a-time loop, which left each scheduler with one latency-bound warp), the per-channel scale / shift are fetched
// from shared memory once per pair, and the vertical half of the pool is a register-to-register maximum.
// (n, row, px) = image, first row of the pair, pixel column of this thread.
template <bool FUSED, bool STATS = false>
__device__ __forceinline__ void strip_drain_pair(const TcStripParams& p, uint32_t ta, uint32_t tb, int n, int row, int px,
                                                 const float* s_scale, const float* s_shift, const float* s_wd, float head_b,
                                                 int lane, int n0, StripStats* st = nullptr) {
  const size_t opix_a = ((size_t)n * p.H + row) * p.W + px, opix_b = opix_a + p.W;
  const size_t oidx_a = opix_a * p.OC + n0, oidx_b = opix_b * p.OC + n0;
  if constexpr (STATS) {
    // training forward: 16-bit stores + the BatchNorm batch statistics of the stored values (every pixel of a strip is valid)
    __nv_bfloat16* orow_a = p.out + oidx_a;
    __nv_bfloat16* orow_b = p.out + oidx_b;
#pragma unroll
    for (int cb = 0; cb < 2; ++cb) {
      const int c = cb * 32;
      if (c < p.Cout) {
        uint32_t ra[32], rb[32];
        tmem_ld_32x32b_x32(ta + c, ra);
        tmem_ld_32x32b_x32(tb + c, rb);
        tmem_ld_wait();
        uint32_t pka[16], pkb[16];
        bn_relu_pack32_x2(ra, rb, s_scale + c, s_shift + c, p.relu, pka, pkb, p.f16);
        store_pk16(orow_a + c, pka);
        store_pk16(orow_b + c, pkb);
        stats_block(pka, true, st->scr, lane, p.f16, st->s[cb], st->q[cb]);
        stats_block(pkb, true, st->scr, lane, p.f16, st->s[cb], st->q[cb]);
      }
    }
    return;
  }
  if (p.out_f32) {                                       // gradient tensors (dgrad): fp32 stores, row by row
#pragma unroll 1
    for (int rr = 0; rr < 2; ++rr) {
      float* orow_f = reinterpret_cast<float*>(p.out) + (rr ? oidx_b : oidx_a);
      for (int c = 0; c < p.Cout; c += 32) {
        uint32_t r[32];
        tmem_ld_32x32b_x32((rr ? tb : ta) + c, r);
        tmem_ld_wait();
#pragma unroll
        for (int q0 = 0; q0 < 32; q0 += 8) {
          uint32_t v[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            float f = fmaf(__uint_as_float(r[q0 + q]), s_scale[c + q0 + q], s_shift[c + q0 + q]);
            if (p.relu) f = fmaxf(f, 0.f);
            v[q] = __float_as_uint(f);
          }
          st_global_v8(orow_f + c + q0, v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7]);
        }
      }
    }
  } else {
    __nv_bfloat16* orow_a = p.out + oidx_a;
    __nv_bfloat16* orow_b = p.out + oidx_b;
    float zacc_a = head_b, zacc_b = head_b;
    for (int c = 0; c < p.Cout; c += 32) {
      uint32_t ra[32], rb[32];
      tmem_ld_32x32b_x32(ta + c, ra);
      tmem_ld_32x32b_x32(tb + c, rb);
      tmem_ld_wait();
      if (FUSED && p.head_kernel && !p.need_y && !p.pool_out) {
        // dec0b at inference: the activation is consumed by the 1x1 head only and never stored, so it is not
        // rounded to 16 bits either: BN + ReLU + dot product stay in (packed) fp32
        float2 za0 = make_float2(0.f, 0.f), za1 = make_float2(0.f, 0.f), zb0 = za0, zb1 = za0;
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          const float4 sc = *reinterpret_cast<const float4*>(s_scale + c + 4 * g);
          const float4 sh = *reinterpret_cast<const float4*>(s_shift + c + 4 * g);
          const float4 wd = *reinterpret_cast<const float4*>(s_wd + c + 4 * g);
          const float2 sc0 = make_float2(sc.x, sc.y), sc1 = make_float2(sc.z, sc.w);
          const float2 sh0 = make_float2(sh.x, sh.y), sh1 = make_float2(sh.z, sh.w);
          float2 a0 = ffma2(make_float2(__uint_as_float(ra[4 * g]), __uint_as_float(ra[4 * g + 1])), sc0, sh0);
          float2 a1 = ffma2(make_float2(__uint_as_float(ra[4 * g + 2]), __uint_as_float(ra[4 * g + 3])), sc1, sh1);
          float2 b0 = ffma2(make_float2(__uint_as_float(rb[4 * g]), __uint_as_float(rb[4 * g + 1])), sc0, sh0);
          float2 b1 = ffma2(make_float2(__uint_as_float(rb[4 * g + 2]), __uint_as_float(rb[4 * g + 3])), sc1, sh1);
          if (p.relu) {
            a0.x = fmaxf(a0.x, 0.f); a0.y = fmaxf(a0.y, 0.f); a1.x = fmaxf(a1.x, 0.f); a1.y = fmaxf(a1.y, 0.f);
            b0.x = fmaxf(b0.x, 0.f); b0.y = fmaxf(b0.y, 0.f); b1.x = fmaxf(b1.x, 0.f); b1.y = fmaxf(b1.y, 0.f);
          }
          za0 = ffma2(a0, make_float2(wd.x, wd.y), za0);
          za1 = ffma2(a1, make_float2(wd.z, wd.w), za1);
          zb0 = ffma2(b0, make_float2(wd.x, wd.y), zb0);
          zb1 = ffma2(b1, make_float2(wd.z, wd.w), zb1);
        }
        zacc_a += (za0.x + za0.y) + (za1.x + za1.y);
        zacc_b += (zb0.x + zb0.y) + (zb1.x + zb1.y);
        continue;
      }
      uint32_t pka[16], pkb[16];
      bn_relu_pack32_x2(ra, rb, s_scale + c, s_shift + c, p.relu, pka, pkb, p.f16);
      if (FUSED && p.head_kernel) {     // head on the rounded (stored) values, four partial sums per row
        float za[4] = {0.f, 0.f, 0.f, 0.f}, zb[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          const float4 wd = *reinterpret_cast<const float4*>(s_wd + c + 4 * g);
          const float2 f0 = unpack16x2(pka[2 * g], p.f16), f1 = unpack16x2(pka[2 * g + 1], p.f16);
          const float2 g0 = unpack16x2(pkb[2 * g], p.f16), g1 = unpack16x2(pkb[2 * g + 1], p.f16);
          za[0] = fmaf(f0.x, wd.x, za[0]); za[1] = fmaf(f0.y, wd.y, za[1]);
          za[2] = fmaf(f1.x, wd.z, za[2]); za[3] = fmaf(f1.y, wd.w, za[3]);
          zb[0] = fmaf(g0.x, wd.x, zb[0]); zb[1] = fmaf(g0.y, wd.y, zb[1]);
          zb[2] = fmaf(g1.x, wd.z, zb[2]); zb[3] = fmaf(g1.y, wd.w, zb[3]);
        }
        zacc_a += (za[0] + za[1]) + (za[2] + za[3]);
        zacc_b += (zb[0] + zb[1]) + (zb[2] + zb[3]);
      }
      if (!FUSED || p.need_y) {
        store_pk16(orow_a + c, pka);
        store_pk16(orow_b + c, pkb);
      }
      if (FUSED && p.pool_out) {
        // 2x2 max-pool (unet_2d_summary.py:176-194): the vertical partner is the other row of the pair, the
        // horizontal partner the neighbouring lane.  The two lanes of a window split the 32 channels: each sends
        // the half its partner will store and keeps the other one - 8 shuffles and one full 32-byte sector per lane.
        const bool odd = (lane & 1) != 0;
        uint32_t mx[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const uint32_t lo = max16x2(pka[q], pkb[q], p.f16), hi = max16x2(pka[8 + q], pkb[8 + q], p.f16);
          const uint32_t got = __shfl_xor_sync(0xffffffffu, odd ? lo : hi, 1);
          mx[q] = max16x2(odd ? hi : lo, got, p.f16);
        }
        __nv_bfloat16* prow = p.pool_out + ((((size_t)n * (p.H >> 1) + (row >> 1)) * (p.W >> 1) + (px >> 1)) * p.Cout
                                            + c + (odd ? 16 : 0));
        st_global_v8(prow, mx[0], mx[1], mx[2], mx[3], mx[4], mx[5], mx[6], mx[7]);
      }
    }
    if (FUSED && p.head_kernel) {
      if (p.logit) { p.logit[opix_a] = zacc_a; p.logit[opix_b] = zacc_b; }
      if (p.prob) { p.prob[opix_a] = 1.f / (1.f + __expf(-zacc_a)); p.prob[opix_b] = 1.f / (1.f + __expf(-zacc_b)); }
    }
  }
}

// Roles: warp 0 = TMA producer, warp 1 = single-thread MMA issuer, warps 2..9 = two epilogue quartets (a quartet
// drains a pair of consecutive 128-pixel tiles, then skips the other quartet's pair).
// FOLD (Cout 32 or 64, normal orientation): an MMA costs the issuing thread ~60 cycles whatever its N is
// (profiles/r1_umma_fold_probe.log), so these layers are issue-rate bound at 9*K/16 MMAs per tile.  Folded mode turns
// the loop inside out: TMEM holds a ring of 512/Cout row accumulators (one per OUTPUT row), and each INPUT halo row i
// is multiplied ONCE per (dx, k) against the stacked weights [W(dy=+1) | W(dy=0) | W(dy=-1)] (N = 3*Cout), which
// accumulates into the three neighbouring accumulators of output rows i-1, i, i+1 at the same time: 3x fewer MMAs,
// every halo row is read from shared memory by 3*K/16 instead of 9*K/16 MMAs.  Output row o is complete once input
// row o+1 has been issued.
template <bool FUSED, bool FOLD, bool STATS = false>
__global__ void __launch_bounds__(ST_THREADS, 1)
tapgemm_tc_strip_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
                        const __grid_constant__ CUtensorMap mapT0, const __grid_constant__ CUtensorMap mapT1,
                        const __grid_constant__ CUtensorMap mapB, const TcStripParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ uint64_t bar_w, row_full[ST_MAX_RING], row_empty[ST_MAX_RING], bar_tfull[16], bar_tempty[16];
  __shared__ uint32_t tmem_base_smem;
  __shared__ __align__(16) float s_scale[128], s_shift[128], s_wd[128];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  StripStats sst;                                                // STATS: this lane's sums (see stats_epilogue.cuh)
  sst.s[0] = sst.s[1] = sst.q[0] = sst.q[1] = make_float2(0.f, 0.f); sst.scr = nullptr;
  if (threadIdx.x == 0) pdl_trigger();
  const int nclu = (FOLD && p.nclu > 1) ? p.nclu : 1;
  const uint32_t crank = nclu > 1 ? cluster_ctarank() : 0u;
  const int n0 = p.n0 + (int)crank * p.Cout;                     // first output channel of THIS CTA
  const int PX = p.swap ? 256 : 128;                             // pixels per tile (one image-row segment)
  // 1024-byte alignment as an offset into the __shared__ array (an integer round trip would turn every later access
  // through this pointer into a generic-space load/store)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int K = p.C0 + p.C1;
  const uint32_t wblk_bytes = p.Cout * p.BK * 2;                 // one (tap, kc) weight tile
  const uint32_t w_bytes = 9u * p.nkc * wblk_bytes;
  uint8_t* s_w = smem;
  uint8_t* s_ring = smem + ((w_bytes + 1023) & ~1023u);
  const uint32_t row_bytes = (uint32_t)p.nkc * p.slot_bytes;     // one halo row = nkc chunk boxes
  uint8_t* s_stage = s_ring + (size_t)p.ring * row_bytes;        // swapped mode only: 4 x 4 KB transpose tiles behind the ring
  const uint32_t box_bytes = (uint32_t)(PX + 2) * p.BK * 2u;
  const int acc_cols = p.swap ? 256 : p.Cout;
  // Normal orientation: draining a [128 px x Cout] accumulator (TMEM load latency + convert + stores) takes a warp
  // quartet ~2x longer than the tensor pipe needs to fill it (measured, profiles/r1_strip_scaling.txt), so TWO
  // quartets drain alternate tile pairs and FOUR accumulator stages keep the pipe busy.  Swapped: 2 x 256 columns.
  // Folded: 512/Cout row accumulators.
  const int nacc = FOLD ? 512 / p.Cout : (p.swap ? 2 : 4);
  const int nacc_sh = FOLD ? (p.Cout == 32 ? 4 : 3) : (p.swap ? 1 : 2), nsets = p.swap ? 1 : ST_QUARTETS;
  uint32_t tmem_cols = 32;
  while (tmem_cols < (uint32_t)(nacc * acc_cols)) tmem_cols <<= 1;

  for (int i = threadIdx.x; i < p.Cout; i += blockDim.x) {
    s_scale[i] = p.scale ? p.scale[n0 + i] : 1.f;
    s_shift[i] = p.shift ? p.shift[n0 + i] : 0.f;
    s_wd[i] = p.head_kernel ? p.head_kernel[2 * i + 1] - p.head_kernel[2 * i] : 0.f;
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapA0);
    if (p.C1 > 0) tma_prefetch_desc(&mapA1);
    tma_prefetch_desc(&mapB);
    mbar_init(&bar_w, 1);
    // a ring slot shared by a cluster is free once BOTH CTAs' MMAs have read it (each MMA thread commits to both)
    for (int s = 0; s < p.ring; ++s) { mbar_init(&row_full[s], 1); mbar_init(&row_empty[s], nclu); }
    for (int s = 0; s < nacc; ++s) { mbar_init(&bar_tfull[s], 1); mbar_init(&bar_tempty[s], 4); }
    mbar_fence_init();
  }
  if (warp == 1) { tmem_alloc(&tmem_base_smem, tmem_cols); tmem_relinquish(); }
  tc_fence_before();
  if (nclu > 1) cluster_sync_all();      // the peer's barriers exist before anything is multicast into this CTA
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;

  // Balanced partition: the N * wsegs image columns (H rows each) are laid end to end and cut into gridDim.x runs of
  // equal length (in units of `gran` rows); a CTA walks its run as one or more strips - a strip never crosses a
  // column boundary - so every SM gets the same number of rows (+-1 unit) and one 2-row halo per strip.
  const int units_per_col = (p.H + p.gran - 1) / p.gran;
  const long long units = (long long)p.N * p.wsegs * units_per_col;
  // (the CTAs of a cluster walk the same strips)
  const long long part = blockIdx.x / nclu, nparts = gridDim.x / nclu;
  const long long u_begin = units * part / nparts, u_end = units * (part + 1) / nparts;
  auto next_strip = [&](long long& u, int& n, int& h0, int& rows, int& w0) -> bool {
    if (u >= u_end) return false;
    const int col = (int)(u / units_per_col), hu = (int)(u - (long long)col * units_per_col);
    long long take = units_per_col - hu;
    if (take > u_end - u) take = u_end - u;
    n = col / p.wsegs; w0 = (col - n * p.wsegs) * PX; h0 = hu * p.gran;
    rows = (int)take * p.gran; if (rows > p.H - h0) rows = p.H - h0;
    u += take;
    return true;
  };

  if (warp == 0) {
    if (elect_one()) {
      // resident weights: B tile (tap, kc) = rows [0, Cout) x cols [tap*K + kc*BK, +BK) of the weight matrix
      mbar_arrive_expect_tx(&bar_w, w_bytes);
      for (int tap = 0; tap < 9; ++tap)
        for (int kc = 0; kc < p.nkc; ++kc)
          tma_load_2d(&mapB, &bar_w,
                      s_w + (size_t)(FOLD ? (kc * 3 + tap % 3) * 3 + (2 - tap / 3) : tap * p.nkc + kc) * wblk_bytes,
                      tap * K + kc * p.BK, n0);   // folded: (kc, dx) groups of three stacked tiles, dy = +1, 0, -1
      int pos = 0; uint32_t empty_parity = 0xffffffffu;          // bit i: parity to wait for on row_empty[i]
      const int kc0 = p.C0 / p.BK;
#ifdef DCB_STRIP_TIMING
      unsigned long long pr_acc[2] = {0, 0};
#endif
      const int rows_per_slot = FOLD ? 2 : 1;                    // folded mode: one barrier per pair of halo rows
      const int nslots = FOLD ? p.ring >> 1 : p.ring;
      long long u = u_begin;
      pdl_wait();                // the weights above are static; the activation rows come from the previous kernel
      for (int n, h0, rows, w0; next_strip(u, n, h0, rows, w0);) {
        for (int rr = -1; rr <= rows; ++rr) {
          const int sub = FOLD ? ((rr + 1) & 1) : 0;              // row inside the slot
          if (sub == 0) {
            ST_T(pc0);
            mbar_wait(&row_empty[pos], (empty_parity >> pos) & 1u);
            ST_T(pc1);
#ifdef DCB_STRIP_TIMING
            pr_acc[0] += (unsigned long long)(pc1 - pc0); pr_acc[1] += 1;
#endif
            empty_parity ^= 1u << pos;
            mbar_arrive_expect_tx(&row_full[pos], rows_per_slot * p.nkc * box_bytes);
          }
          uint8_t* dst = s_ring + ((size_t)pos * rows_per_slot + sub) * row_bytes;
          for (int kc = 0; kc < p.nkc; ++kc) {
            const bool second = kc >= kc0;
            const int cc = (second ? kc - kc0 : kc) * p.BK;
            if (nclu > 1) {      // each CTA of the pair fetches every other channel chunk and multicasts it into both
              if ((kc & 1) == (int)crank)
                tma_load_4d_mc(second ? &mapA1 : &mapA0, &row_full[pos], dst + (size_t)kc * p.slot_bytes, cc, w0 - 1, h0 + rr, n, 3);
              continue;
            }
            tma_load_4d(second ? &mapA1 : &mapA0, &row_full[pos], dst + (size_t)kc * p.slot_bytes, cc, w0 - 1, h0 + rr, n);
            if (p.swap)   // 258-pixel halo row = a 256-pixel box + a 2-pixel box (TMA boxes are limited to 256 per dim)
              tma_load_4d(second ? &mapT1 : &mapT0, &row_full[pos], dst + (size_t)kc * p.slot_bytes + 256u * p.BK * 2u, cc,
                          w0 + 255, h0 + rr, n);
          }
          if (sub == rows_per_slot - 1 && ++pos == nslots) pos = 0;
        }
      }
#ifdef DCB_STRIP_TIMING
      g_strip_dbg2[blockIdx.x * 16 + 0] = pr_acc[0]; g_strip_dbg2[blockIdx.x * 16 + 1] = pr_acc[1];
#endif
    }
  } else if (warp == 1) {
    if (elect_one()) {
      const uint32_t idesc = p.swap ? make_idesc_16(128, 256, 0, 0, p.f16) : make_idesc_16(TC_BM, p.Cout, 0, 0, p.f16);
      const uint32_t swz = (p.BK == 64) ? SWZ_128B : SWZ_64B;
      const uint32_t pitch = p.BK * 2u, sbo = 8u * pitch;
      const int ksteps = p.BK / 16;
      const uint64_t dbase = make_smem_desc(0, 16, sbo, swz);
      const uint32_t ring16 = smem_u32(s_ring) >> 4, w16 = smem_u32(s_w) >> 4, rowb16 = row_bytes >> 4;
      const uint32_t slot16 = (uint32_t)p.slot_bytes >> 4, pitch16 = pitch >> 4, wblk16 = wblk_bytes >> 4;
      mbar_wait(&bar_w, 0);
      tc_fence_after();
      int pos_next = 0; uint32_t full_parity = 0;                // bit i: parity to wait for on row_full[i]
      auto wait_next_row = [&]() -> int {
        const int ps = pos_next;
        mbar_wait(&row_full[ps], (full_parity >> ps) & 1u);
        full_parity ^= 1u << ps;
        pos_next = (ps + 1 == p.ring) ? 0 : ps + 1;
        return ps;
      };
      uint32_t j = 0;                                            // tile counter of this CTA
      if constexpr (FOLD) {
        // Synchronisation is per PAIR of rows: every mbarrier wait / tcgen05.commit costs the issuing thread a few
        // hundred cycles (profiles/r1_umma_overhead_probe.log), as much as the 7 MMAs of a row.  Input rows (2m-1, 2m)
        // arrive under one row_full barrier, open the output pair P(m) = rows (2m, 2m+1) (one tempty barrier, armed by the
        // epilogue quartet that drains that pair) and complete the pair P(m-1) (one tfull commit).
        const uint32_t id0 = make_idesc_16(TC_BM, 0, 0, 0, p.f16), idu = ((uint32_t)p.Cout >> 3) << 17;   // N field += Cout per row
        const uint32_t nmask = (uint32_t)nacc - 1u, pmask = ((uint32_t)nacc >> 1) - 1u;
        const int pair_sh = nacc_sh - 1;
        const uint64_t dW = dbase + w16;
        const uint32_t a_row_full = smem_u32_pinned(row_full), a_row_empty = smem_u32_pinned(row_empty);
        const uint32_t a_tfull = smem_u32_pinned(bar_tfull), a_tempty = smem_u32_pinned(bar_tempty);
        const int ring_pairs = p.ring >> 1;
        int pp = 0; uint32_t fullpar = 0;
        asm volatile(".reg .pred p_rf, p_te;");                   // split-phase poll results, see the pair loop
#ifdef DCB_STRIP_TIMING
        unsigned long long dbg_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        const long long dbg_t0 = clock64();
#endif
        // halo row i of the current strip (rows output rows, first output row = tile j) -> output rows [i-1, i+1]
        auto issue_row_generic = [&](int i, int rows, uint64_t dA) {
          const bool opens = i + 1 < rows;                        // output row i+1 receives its first contribution
          // the weight tile of output row o inside a (kc, dx) group is o - i + 1; the accumulator ring may wrap inside
          // the span: one or two MMAs (segments) per step
          const int o_lo = i - 1 < 0 ? 0 : i - 1, o_hi = i + 1 < rows ? i + 1 : rows - 1;
          const uint32_t sa = (j + (uint32_t)o_lo) & nmask;
          const int t0 = o_lo - i + 1;
          {   // first step (kc = 0, dx = 0, k = 0): a newly opened row starts with accumulate = 0
            const int cnt = (opens ? i : o_hi) - o_lo + 1;        // rows that are already open
            const int run = cnt < (int)(nacc - sa) ? cnt : (int)(nacc - sa);
            if (run > 0) umma_bf16(tmem_base + sa * (uint32_t)p.Cout, dA, dW + (uint32_t)t0 * wblk16, id0 + run * idu, 1u);
            if (run < cnt) umma_bf16(tmem_base, dA, dW + (uint32_t)(t0 + run) * wblk16, id0 + (cnt - run) * idu, 1u);
            if (opens)
              umma_bf16(tmem_base + ((j + (uint32_t)(i + 1)) & nmask) * (uint32_t)p.Cout, dA, dW + 2u * wblk16, id0 + idu, 0u);
          }
          const int cnt = o_hi - o_lo + 1;
          const int run = cnt < (int)(nacc - sa) ? cnt : (int)(nacc - sa);
          const uint32_t d0 = tmem_base + sa * (uint32_t)p.Cout, idesc0 = id0 + run * idu;
          const uint64_t dW0 = dW + (uint32_t)t0 * wblk16;
          if (run == cnt) {
            if (ksteps == 4) fold_issue_rest<4, false>(d0, 0, dA, dW0, 0, idesc0, 0, p.nkc, slot16, pitch16, wblk16);
            else fold_issue_rest<2, false>(d0, 0, dA, dW0, 0, idesc0, 0, p.nkc, slot16, pitch16, wblk16);
          } else {
            const uint64_t dW1 = dW + (uint32_t)(t0 + run) * wblk16;
            const uint32_t idesc1 = id0 + (cnt - run) * idu;
            if (ksteps == 4) fold_issue_rest<4, true>(d0, tmem_base, dA, dW0, dW1, idesc0, idesc1, p.nkc, slot16, pitch16, wblk16);
            else fold_issue_rest<2, true>(d0, tmem_base, dA, dW0, dW1, idesc0, idesc1, p.nkc, slot16, pitch16, wblk16);
          }
        };
        long long u = u_begin;
        for (int n, h0, rows, w0; next_strip(u, n, h0, rows, w0);) {
          const int half = rows >> 1;                             // rows is even in folded mode
          // Split-phase barrier polls: a phase check costs this thread ~250 cycles of latency even when the phase is
          // long complete, so the two checks of pair m+1 are ISSUED (non-blocking mbarrier.test_wait into the
          // function-scope predicates p_rf / p_te) before the MMAs of pair m and only CONSUMED at the top of the next
          // iteration; a poll that came back "not yet" falls back to the blocking wait.
          bool pre = false, pre_te = false;
          for (int m = 0; m <= half; ++m) {                       // input (halo) rows h0 + 2m - 1 and h0 + 2m
            ST_T(c0);
            ST_DECL(c1);
            const uint32_t jp = (j >> 1) + (uint32_t)m;           // running index of the output pair P(m)
            {
              uint32_t ok_rf = 0, ok_te = 0;
              if (pre) {
                asm volatile("selp.u32 %0, 1, 0, p_rf;" : "=r"(ok_rf));
                if (pre_te) asm volatile("selp.u32 %0, 1, 0, p_te;" : "=r"(ok_te));
              }
              if (!ok_rf) mbar_wait_a(a_row_full + 8u * pp, (fullpar >> pp) & 1u);
              fullpar ^= 1u << pp;
              ST_SET(c1); ST_ACC(0, c0, c1);
              if (m < half && !ok_te) mbar_wait_a(a_tempty + 8u * (jp & pmask), ((jp >> pair_sh) & 1u) ^ 1u);
            }
            tc_fence_after();
            ST_T(c2); ST_ACC(1, c1, c2);
            pre = m < half;
            pre_te = m + 1 < half;
            if (pre) {
              const int ppn = (pp + 1 == ring_pairs) ? 0 : pp + 1;
              asm volatile("mbarrier.test_wait.parity.shared::cta.b64 p_rf, [%0], %1;" ::"r"(a_row_full + 8u * ppn),
                           "r"((fullpar >> ppn) & 1u) : "memory");
              if (pre_te)
                asm volatile("mbarrier.test_wait.parity.shared::cta.b64 p_te, [%0], %1;" ::"r"(a_tempty + 8u * ((jp + 1u) & pmask)),
                             "r"((((jp + 1u) >> pair_sh) & 1u) ^ 1u) : "memory");
            }
            const uint64_t dA0 = dbase + (ring16 + (uint32_t)pp * 2u * rowb16), dA1 = dA0 + rowb16;
            if (m >= 1 && m < half && (jp & pmask) != 0u) {        // interior pair, its four accumulators are contiguous
              const uint32_t d0 = tmem_base + (((jp - 1u) & pmask) * 2u) * (uint32_t)p.Cout, C = (uint32_t)p.Cout;
              if (ksteps == 4) {
                fold_issue_fast<4>(d0, d0 + 2u * C, dA0, dW, id0 + idu, id0 + 2u * idu, id0 + 3u * idu, p.nkc, slot16, pitch16, wblk16);
                fold_issue_fast<4>(d0 + C, d0 + 3u * C, dA1, dW, id0 + idu, id0 + 2u * idu, id0 + 3u * idu, p.nkc, slot16, pitch16, wblk16);
              } else {
                fold_issue_fast<2>(d0, d0 + 2u * C, dA0, dW, id0 + idu, id0 + 2u * idu, id0 + 3u * idu, p.nkc, slot16, pitch16, wblk16);
                fold_issue_fast<2>(d0 + C, d0 + 3u * C, dA1, dW, id0 + idu, id0 + 2u * idu, id0 + 3u * idu, p.nkc, slot16, pitch16, wblk16);
              }
#ifdef DCB_STRIP_TIMING
              dbg_acc[5] += 1;
#endif
            } else {
              issue_row_generic(2 * m - 1, rows, dA0);
              issue_row_generic(2 * m, rows, dA1);
            }
            ST_T(c3); ST_ACC(2, c2, c3);
            if (nclu > 1) umma_commit_mc2(a_row_empty + 8u * pp);                 // the slot is shared with the peer CTA
            else umma_commit_a(a_row_empty + 8u * pp);
            if (m >= 1) umma_commit_a(a_tfull + 8u * ((jp - 1u) & pmask));       // output pair P(m-1) is complete
            ST_T(c4); ST_ACC(3, c3, c4); ST_ACC(4, c0, c4);
            if (++pp == ring_pairs) pp = 0;
          }
          j += (uint32_t)rows;
        }
#ifdef DCB_STRIP_TIMING
        dbg_acc[6] = (unsigned long long)(clock64() - dbg_t0);
        for (int q = 0; q < 8; ++q) g_strip_dbg[blockIdx.x * 8 + q] = dbg_acc[q];
#endif
      } else {
      long long u = u_begin;
      for (int n, h0, rows, w0; next_strip(u, n, h0, rows, w0);) {
        int p0 = wait_next_row(), p1 = wait_next_row();          // halo rows h0-1 and h0
        for (int t = 0; t < rows; ++t, ++j) {
          const int p2 = wait_next_row();                         // halo row h0+t+1
          const int acc = j & (nacc - 1);
          const uint32_t acc_phase = (j >> nacc_sh) & 1u;
          mbar_wait(&bar_tempty[acc], acc_phase ^ 1);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + (uint32_t)(acc * acc_cols);
          const uint32_t row16[3] = {ring16 + p0 * rowb16, ring16 + p1 * rowb16, ring16 + p2 * rowb16};
          if (p.swap) {
            if (ksteps == 4) strip_issue_tile<4, true>(d_tmem, dbase, row16, w16, p.nkc, slot16, pitch16, wblk16, idesc);
            else strip_issue_tile<2, true>(d_tmem, dbase, row16, w16, p.nkc, slot16, pitch16, wblk16, idesc);
          } else {
            if (ksteps == 4) strip_issue_tile<4, false>(d_tmem, dbase, row16, w16, p.nkc, slot16, pitch16, wblk16, idesc);
            else strip_issue_tile<2, false>(d_tmem, dbase, row16, w16, p.nkc, slot16, pitch16, wblk16, idesc);
          }
          umma_commit(&bar_tfull[acc]);
          umma_commit(&row_empty[p0]);                            // halo row t is not needed by later tiles
          p0 = p1; p1 = p2;
        }
        umma_commit(&row_empty[p0]);
        umma_commit(&row_empty[p1]);
      }
      }
    }
  } else {
    const int quarter = warp & 3;
    const int eset = (warp - 2) >> 2;                            // epilogue quartet: drains the tile pairs (j >> 1) % nsets == eset
    const int m = quarter * 32 + lane;
#ifdef DCB_STRIP_TIMING
    long long ep_last = 0;
    unsigned long long ep_acc[5] = {0, 0, 0, 0, 0};
#endif
    const float head_b = (FUSED && p.head_kernel) ? (p.head_bias[1] - p.head_bias[0]) : 0.f;   // hoisted: two global loads
    uint32_t pool_prev[2][16];                                   // previous row (bf16 pairs) for the fused 2x2 max-pool
#pragma unroll
    for (int q = 0; q < 16; ++q) { pool_prev[0][q] = 0; pool_prev[1][q] = 0; }
    uint32_t j = 0;
    long long u = u_begin;
    if constexpr (FOLD) {
      // Folded mode hands the epilogue PAIRS of output rows (one tfull / tempty barrier per pair, see the MMA warp): a
      // quartet drains both rows of its pair together (strip_drain_pair).
      if constexpr (STATS) sst.scr = reinterpret_cast<uint32_t*>(s_stage) + (warp - 2) * STATS_SCRATCH_WORDS;
      const uint32_t t_lane = tmem_base + ((uint32_t)(quarter * 32) << 16);
      const uint32_t pmask = ((uint32_t)nacc >> 1) - 1u;
      for (int n, h0, rows, w0; next_strip(u, n, h0, rows, w0);) {
        for (int t = 0; t < rows; t += 2, j += 2) {
          const uint32_t jp = j >> 1;
          if ((int)(jp & 1u) != eset) continue;                  // ST_QUARTETS == 2: alternate pairs
          const uint32_t ta = t_lane + (j & (uint32_t)(nacc - 1)) * (uint32_t)p.Cout, tb = ta + (uint32_t)p.Cout;
          const int bar_i = (int)(jp & pmask);
          mbar_wait(&bar_tfull[bar_i], (j >> nacc_sh) & 1u);
          tc_fence_after();
          strip_drain_pair<FUSED, STATS>(p, ta, tb, n, h0 + t, w0 + m, s_scale, s_shift, s_wd, head_b, lane, n0, &sst);
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&bar_tempty[bar_i]);
        }
      }
    } else
    for (int n, h0, rows, w0; eset < nsets && next_strip(u, n, h0, rows, w0);) {
      for (int t = 0; t < rows; ++t, ++j) {
        if ((int)((j >> 1) % (uint32_t)nsets) != eset) continue;
        const int acc = j & (nacc - 1);
        const uint32_t acc_phase = (j >> nacc_sh) & 1u;
        // folded mode: the barriers are per PAIR of tiles (see the MMA warp); wait before the even tile, arrive after the odd one
        const int bar_i = FOLD ? (int)((j >> 1) & (uint32_t)((nacc >> 1) - 1)) : acc;
        const uint32_t bar_phase = FOLD ? ((j >> nacc_sh) & 1u) : acc_phase;
        const bool do_wait = !FOLD || (j & 1u) == 0u, do_arrive = !FOLD || (j & 1u) != 0u;
        if (p.swap) {
          const bool warp_valid = quarter * 32 < p.Cout;
          const float sc = warp_valid ? s_scale[quarter * 32 + lane] : 0.f, sh = warp_valid ? s_shift[quarter * 32 + lane] : 0.f;
          const size_t row0 = (((size_t)n * p.H + (h0 + t)) * p.W + w0) * p.OC + p.n0 + quarter * 32;
          auto pix_index = [&](int mm) -> long long { return (long long)(row0 + (size_t)mm * p.OC); };
          mbar_wait(&bar_tfull[acc], acc_phase);
          tc_fence_after();
          epilogue_swapped(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * acc_cols), 256, warp_valid, sc, sh,
                           p.relu, p.out_f32, p.out, s_stage + quarter * 4096, lane, pix_index, p.f16);
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&bar_tempty[acc]);
          continue;
        }
        if constexpr (!FUSED) {
          const size_t oidx = (((size_t)n * p.H + (h0 + t)) * p.W + (w0 + m)) * p.OC + p.n0;
          __nv_bfloat16* orow = p.out + oidx;
          float* orow_f = reinterpret_cast<float*>(p.out) + oidx;
          ST_T(ec0);
          if (do_wait) mbar_wait(&bar_tfull[bar_i], bar_phase);
          tc_fence_after();
          ST_T(ec1);
#ifdef DCB_STRIP_TIMING
          ep_acc[0] += (unsigned long long)(ec1 - ec0); ep_acc[1] += 1;
          if (ep_last) ep_acc[2] += (unsigned long long)(ec0 - ep_last);
          ep_last = ec1;
#endif
          const uint32_t t_addr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * p.Cout);
          for (int c = 0; c < p.Cout; c += 32) {
            uint32_t r[32];
            ST_T(lc0);
            tmem_ld_32x32b_x32(t_addr + c, r);
            tmem_ld_wait();
            ST_T(lc1);
#ifdef DCB_STRIP_TIMING
            ep_acc[3] += (unsigned long long)(lc1 - lc0);
#endif
            if (p.out_f32) {
  #pragma unroll
              for (int j = 0; j < 32; j += 8) {
                uint32_t v[8];
  #pragma unroll
                for (int q = 0; q < 8; ++q) {
                  float f = fmaf(__uint_as_float(r[j + q]), s_scale[c + j + q], s_shift[c + j + q]);
                  if (p.relu) f = fmaxf(f, 0.f);
                  v[q] = __float_as_uint(f);
                }
                st_global_v8(orow_f + c + j, v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7]);
              }
            } else {
              uint32_t pk[16];
              bn_relu_pack32(r, s_scale + c, s_shift + c, p.relu, pk, p.f16);
              store_pk16(orow + c, pk);
            }
#ifdef DCB_STRIP_TIMING
            { const long long lc2 = clock64(); ep_acc[4] += (unsigned long long)(lc2 - lc1); }
#endif
          }
        } else {
          const size_t opix = ((size_t)n * p.H + (h0 + t)) * p.W + (w0 + m);
          const size_t oidx = opix * p.Cout;
          __nv_bfloat16* orow = p.out + oidx;
          float* orow_f = reinterpret_cast<float*>(p.out) + oidx;
          ST_T(ec0);
          if (do_wait) mbar_wait(&bar_tfull[bar_i], bar_phase);
          tc_fence_after();
          ST_T(ec1);
#ifdef DCB_STRIP_TIMING
          ep_acc[0] += (unsigned long long)(ec1 - ec0); ep_acc[1] += 1;
          if (ep_last) ep_acc[2] += (unsigned long long)(ec0 - ep_last);
          ep_last = ec1;
#endif
          const uint32_t t_addr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * p.Cout);
          float zacc = head_b;
  #pragma unroll
          for (int cb = 0; cb < 4; ++cb) {
            const int c = cb * 32;
            if (c >= p.Cout) break;
            uint32_t r[32];
            tmem_ld_32x32b_x32(t_addr + c, r);
            tmem_ld_wait();
            if (p.out_f32) {
  #pragma unroll
              for (int j = 0; j < 32; j += 8) {
                uint32_t v[8];
  #pragma unroll
                for (int q = 0; q < 8; ++q) {
                  float f = fmaf(__uint_as_float(r[j + q]), s_scale[c + j + q], s_shift[c + j + q]);
                  if (p.relu) f = fmaxf(f, 0.f);
                  v[q] = __float_as_uint(f);
                }
                st_global_v8(orow_f + c + j, v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7]);
              }
            } else if (p.head_kernel && !p.need_y && !p.pool_out) {
              // dec0b at inference: the activation is consumed by the 1x1 head only and never stored, so it is not
              // rounded to bf16 either: BN + ReLU + dot product stay in (packed) fp32
              float2 za0 = make_float2(0.f, 0.f), za1 = make_float2(0.f, 0.f);
  #pragma unroll
              for (int g = 0; g < 8; ++g) {
                const float4 sc = *reinterpret_cast<const float4*>(s_scale + c + 4 * g);
                const float4 sh = *reinterpret_cast<const float4*>(s_shift + c + 4 * g);
                const float4 wd = *reinterpret_cast<const float4*>(s_wd + c + 4 * g);
                float2 v0 = ffma2(make_float2(__uint_as_float(r[4 * g]), __uint_as_float(r[4 * g + 1])), make_float2(sc.x, sc.y),
                                  make_float2(sh.x, sh.y));
                float2 v1 = ffma2(make_float2(__uint_as_float(r[4 * g + 2]), __uint_as_float(r[4 * g + 3])), make_float2(sc.z, sc.w),
                                  make_float2(sh.z, sh.w));
                if (p.relu) { v0.x = fmaxf(v0.x, 0.f); v0.y = fmaxf(v0.y, 0.f); v1.x = fmaxf(v1.x, 0.f); v1.y = fmaxf(v1.y, 0.f); }
                za0 = ffma2(v0, make_float2(wd.x, wd.y), za0);
                za1 = ffma2(v1, make_float2(wd.z, wd.w), za1);
              }
              zacc += (za0.x + za0.y) + (za1.x + za1.y);
            } else {
              uint32_t pk[16];
              bn_relu_pack32(r, s_scale + c, s_shift + c, p.relu, pk, p.f16);
              if (p.head_kernel) {            // head on the rounded (stored) bf16 values, four partial sums
                float za[4] = {0.f, 0.f, 0.f, 0.f};
  #pragma unroll
                for (int g = 0; g < 8; ++g) {
                  const float4 wd = *reinterpret_cast<const float4*>(s_wd + c + 4 * g);
                  const float2 f0 = unpack16x2(pk[2 * g], p.f16);
                  const float2 f1 = unpack16x2(pk[2 * g + 1], p.f16);
                  za[0] = fmaf(f0.x, wd.x, za[0]); za[1] = fmaf(f0.y, wd.y, za[1]);
                  za[2] = fmaf(f1.x, wd.z, za[2]); za[3] = fmaf(f1.y, wd.w, za[3]);
                }
                zacc += (za[0] + za[1]) + (za[2] + za[3]);
              }
              if (p.need_y) {
                store_pk16(orow + c, pk);
              }
              if (p.pool_out && cb < 2) {
                // 2x2 max-pool: vertical partner = the previous tile of this warp (row h0+t-1, kept in registers),
                // horizontal partner = the neighbouring lane.  R and H are even, so pairs never straddle work items.
                if ((t & 1) == 0) {
  #pragma unroll
                  for (int q = 0; q < 16; ++q) pool_prev[cb][q] = pk[q];
                } else {
                  uint32_t mx[16];
  #pragma unroll
                  for (int q = 0; q < 16; ++q) {
                    const uint32_t au = max16x2(pk[q], pool_prev[cb][q], p.f16);
                    const uint32_t bu = __shfl_xor_sync(0xffffffffu, au, 1);
                    mx[q] = max16x2(au, bu, p.f16);
                  }
                  if ((lane & 1) == 0) {
                    __nv_bfloat16* prow = p.pool_out + ((((size_t)n * (p.H >> 1) + ((h0 + t) >> 1)) * (p.W >> 1) + ((w0 + m) >> 1)) * p.Cout + c);
                    store_pk16(prow, mx);
                  }
                }
              }
            }
          }
          if (p.head_kernel) {
            if (p.logit) p.logit[opix] = zacc;
            if (p.prob) p.prob[opix] = 1.f / (1.f + __expf(-zacc));
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0 && do_arrive) mbar_arrive(&bar_tempty[bar_i]);
      }
    }
#ifdef DCB_STRIP_TIMING
    if (lane == 0 && quarter == 0 && eset < 2)
      for (int q = 0; q < 5; ++q) g_strip_dbg2[blockIdx.x * 16 + 2 + 5 * eset + q] = ep_acc[q];
#endif
  }
  tc_fence_before();
  if (nclu > 1) cluster_sync_all();      // the peer may still multicast into this CTA / commit to its barriers until here
  else __syncthreads();
  if (warp == 1) { tc_fence_after(); tmem_dealloc(tmem_base, tmem_cols); }
  if constexpr (STATS) {
    // every MMA has retired: the halo ring takes the per-warp accumulators ([8 warps][nblk][16][4] floats)
    float* dump = reinterpret_cast<float*>(s_ring);
    const int nblk = p.Cout / 32;
    if (warp >= 2 && lane < 16) {
#pragma unroll
      for (int bi = 0; bi < 2; ++bi)
        if (bi < nblk)
          *reinterpret_cast<float4*>(dump + ((size_t)((warp - 2) * nblk + bi) * 16 + lane) * 4) =
              make_float4(sst.s[bi].x, sst.s[bi].y, sst.q[bi].x, sst.q[bi].y);
    }
    __syncthreads();
    stats_cta_finish(dump, 8, nblk, [](int bi) { return bi * 32; }, p.Cout, p.stat_sums);
  }
}

// ====================================================================================== CTA-pair folded strip kernel
// The folded strip loop on PAIR MMAs (tcgen05 cta_group::2, a cluster of two CTAs on neighbouring SMs): one instruction
// multiplies M = 256 pixels - the 128-pixel halo row segment of each CTA, read from that CTA's own shared memory -
// against N = 1..3 x Cout stacked weight rows of which each CTA holds HALF, and accumulates into both CTAs' tensor
// memory.  A single-CTA MMA occupies the tensor pipe for 89-109 cycles whatever N <= 128 is; the pair instruction takes
// 48 cycles at N = 64 and 64 at N = 128 for twice the rows (profiles/r1_umma_cta2_probe.log), so the N = 96 / 192 MMAs
// of the 32- and 64-channel layers - which bound those layers once the epilogue was fixed - cost each SM about half.
//   * The two CTAs of a pair walk the SAME rows of two neighbouring 128-pixel columns in lockstep.  Each runs its own TMA
//     producer (its halo rows into its own ring, byte counts signalled on the LEADER's row_full barrier through the
//     .cta_group::2 form of the bulk-tensor load) and its own epilogue quartets (arriving on the leader's tempty barrier
//     with a cluster-scope remote arrive); the leader's single MMA thread issues for both and multicasts its commits
//     (row_empty, tfull) to both CTAs' barriers.
//   * Weights: for a span of `run` output rows starting at stacked tile t0 the instruction reads N/2 = run * Cout / 2
//     rows at ONE descriptor offset from each CTA - rows [t0*Cout, +N/2) of the stack from the leader, [t0*Cout + N/2,
//     +N/2) from the peer.  The six (t0, run) spans of the folded loop (2-row accumulate, opening row, 3-row step, and
//     the spans at strip edges / where the accumulator ring wraps) therefore get one region each: 10 half tiles per
//     (kc, dx) group and CTA instead of 6 - 5/3 of the single-CTA footprint, still small for Cout = 32.
// region offset (in half tiles of Cout/2 rows) of span (t0, run) inside a (kc, dx) weight group
__device__ __forceinline__ uint32_t st2_region(int t0, int run) {
  return run == 3 ? 7u : (run == 2 ? (t0 == 0 ? 3u : 5u) : (uint32_t)t0);
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// arrive / arrive.expect_tx on a barrier of any CTA of the cluster (shared::cluster address, e.g. from mapa_u32).
// RELAXED on purpose: the release form at cluster scope compiles to MEMBAR.ALL.GPU + ERRBAR in front of the arrive, i.e.
// every epilogue warp waited for its global stores to be performed before it could hand its accumulators back (40 % of
// all stall samples of the first version, profiles/r2_strip_pair_ncu.txt).  What the arrive has to order is the TMEM
// reads (tcgen05.wait::ld + tcgen05.fence::before_thread_sync in front of it) / nothing at all for the producer.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_addr) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx_cluster(uint32_t bar_addr, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.relaxed.cluster.shared::cluster.b64 _, [%0], %1;" ::"r"(bar_addr), "r"(bytes) : "memory");
}
// bulk-tensor loads whose completion is signalled on a barrier of either CTA of the pair
__device__ __forceinline__ void tma_load_2d_pair(const CUtensorMap* m, uint32_t bar_addr, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.cta_group::2 [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_addr), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_4d_pair(const CUtensorMap* m, uint32_t bar_addr, void* dst, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes.cta_group::2 [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_addr), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// arrives on the barrier at this shared-memory offset in BOTH CTAs once all earlier pair MMAs have completed
__device__ __forceinline__ void umma2_commit_both(uint32_t bar_addr) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar_addr), "h"((uint16_t)3) : "memory");
}

// interior halo row whose three accumulators are contiguous in the ring (cf. fold_issue_fast): rows i-1, i accumulate
// (N = 2*Cout, region (0,2)), row i+1 is opened with accumulate = 0 (N = Cout, region (2,1)); then N = 3*Cout (region (0,3))
template <int KSTEPS>
__device__ __forceinline__ void fold2_issue_fast(uint32_t d0, uint32_t d2, uint64_t dA, uint64_t dW, uint32_t id1, uint32_t id2,
                                                 uint32_t id3, int nkc, uint32_t slot16, uint32_t pitch16, uint32_t half16,
                                                 uint32_t group16) {
  umma2_bf16(d0, dA, dW + 3u * half16, id2, 1u);
  umma2_bf16(d2, dA, dW + 2u * half16, id1, 0u);
  const uint64_t dW3 = dW + 7u * half16;
  for (int kc = 0; kc < nkc; ++kc) {
#pragma unroll
    for (int dx = 0; dx < 3; ++dx) {
#pragma unroll
      for (int k = 0; k < KSTEPS; ++k) {
        if (kc == 0 && dx == 0 && k == 0) continue;
        umma2_bf16(d0, dA + (kc * slot16 + dx * pitch16 + 2 * k), dW3 + ((uint32_t)(kc * 3 + dx) * group16 + 2 * k), id3, 1u);
      }
    }
  }
}

template <bool FUSED>
__global__ void __launch_bounds__(ST_THREADS, 1)
tapgemm_tc_strip2_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
                         const __grid_constant__ CUtensorMap mapBh, const TcStripParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ uint64_t bar_w, row_full[ST_MAX_RING / 2], row_empty[ST_MAX_RING / 2], bar_tfull[8], bar_tempty[8];
  __shared__ uint32_t tmem_base_smem;
  __shared__ __align__(16) float s_scale[128], s_shift[128], s_wd[128];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) pdl_trigger();
  const uint32_t rank = cluster_ctarank();
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int K = p.C0 + p.C1;
  const int hrows = p.Cout >> 1;                                  // rows of a half tile
  const uint32_t half_bytes = (uint32_t)hrows * p.BK * 2u;
  const uint32_t group_bytes = 10u * half_bytes;
  const uint32_t w_bytes = 3u * p.nkc * group_bytes;
  uint8_t* s_w = smem;
  uint8_t* s_ring = smem + ((w_bytes + 1023) & ~1023u);
  const uint32_t row_bytes = (uint32_t)p.nkc * p.slot_bytes;
  const uint32_t box_bytes = 130u * p.BK * 2u;
  const int nacc = 512 / p.Cout, nacc_sh = p.Cout == 32 ? 4 : 3;
  const int ring_pairs = p.ring >> 1;

  for (int i = threadIdx.x; i < p.Cout; i += blockDim.x) {
    s_scale[i] = p.scale ? p.scale[p.n0 + i] : 1.f;
    s_shift[i] = p.shift ? p.shift[p.n0 + i] : 0.f;
    s_wd[i] = p.head_kernel ? p.head_kernel[2 * i + 1] - p.head_kernel[2 * i] : 0.f;
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapA0);
    if (p.C1 > 0) tma_prefetch_desc(&mapA1);
    tma_prefetch_desc(&mapBh);
    // the leader's copies of bar_w / row_full / tempty are the ones in use; both CTAs initialise theirs alike
    mbar_init(&bar_w, 2);
    for (int s = 0; s < ring_pairs; ++s) { mbar_init(&row_full[s], 2); mbar_init(&row_empty[s], 1); }
    for (int s = 0; s < (nacc >> 1); ++s) { mbar_init(&bar_tfull[s], 1); mbar_init(&bar_tempty[s], 8); }
    mbar_fence_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_smem)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;

  // Balanced partition over PAIRS of neighbouring 128-pixel columns (N * wsegs is even): pair q of the grid walks its run
  // of row pairs; CTA `rank` of the pair takes column 2 * pcol + rank
  const int units_per_col = p.H >> 1;
  const int npairs = gridDim.x >> 1, pair = blockIdx.x >> 1;
  const long long units = (long long)(p.N * p.wsegs / 2) * units_per_col;
  const long long u_begin = units * pair / npairs, u_end = units * (pair + 1) / npairs;
  auto next_strip = [&](long long& u, int& n, int& h0, int& rows, int& w0) -> bool {
    if (u >= u_end) return false;
    const int pcol = (int)(u / units_per_col), hu = (int)(u - (long long)pcol * units_per_col);
    long long take = units_per_col - hu;
    if (take > u_end - u) take = u_end - u;
    const int col = 2 * pcol + (int)rank;
    n = col / p.wsegs; w0 = (col - n * p.wsegs) * 128; h0 = hu * 2;
    rows = (int)take * 2;
    u += take;
    return true;
  };

  if (warp == 0) {
    if (elect_one()) {
      const uint32_t l_bar_w = mapa_u32(smem_u32(&bar_w), 0), l_row_full = mapa_u32(smem_u32(row_full), 0);
      // this CTA's halves of the stacked weights: logical half tile ht of a group = rows [(ht & 1) * hrows, +hrows) of the
      // weight matrix at tap (dy = 1 - ht / 2, dx) - stacked in the order dy = +1, 0, -1 like the single-CTA kernel
      mbar_arrive_expect_tx_cluster(l_bar_w, w_bytes);
      for (int kc = 0; kc < p.nkc; ++kc)
        for (int dx = 0; dx < 3; ++dx) {
          uint8_t* g = s_w + (size_t)(kc * 3 + dx) * group_bytes;
          for (int t0 = 0; t0 < 3; ++t0)
            for (int run = 1; run + t0 <= 3; ++run) {
              if (t0 == 2 && run != 1) continue;
              const uint32_t off = st2_region(t0, run);
              for (int e = 0; e < run; ++e) {
                const int ht = 2 * t0 + (int)rank * run + e;
                const int tap = (2 - (ht >> 1)) * 3 + dx;
                tma_load_2d_pair(&mapBh, l_bar_w, g + (size_t)(off + e) * half_bytes, tap * K + kc * p.BK, p.n0 + (ht & 1) * hrows);
              }
            }
        }
      int pos = 0; uint32_t empty_parity = 0xffffffffu;
      const int kc0 = p.C0 / p.BK;
      long long u = u_begin;
      pdl_wait();                // the weights above are static; the activation rows come from the previous kernel
      for (int n, h0, rows, w0; next_strip(u, n, h0, rows, w0);) {
        for (int rr = -1; rr <= rows; ++rr) {
          const int sub = (rr + 1) & 1;
          if (sub == 0) {
            mbar_wait(&row_empty[pos], (empty_parity >> pos) & 1u);
            empty_parity ^= 1u << pos;
            mbar_arrive_expect_tx_cluster(l_row_full + 8u * pos, 2u * p.nkc * box_bytes);
          }
          uint8_t* dst = s_ring + ((size_t)pos * 2 + sub) * row_bytes;
          for (int kc = 0; kc < p.nkc; ++kc) {
            const bool second = kc >= kc0;
            const int cc = (second ? kc - kc0 : kc) * p.BK;
            tma_load_4d_pair(second ? &mapA1 : &mapA0, l_row_full + 8u * pos, dst + (size_t)kc * p.slot_bytes, cc, w0 - 1, h0 + rr, n);
          }
          if (sub == 1 && ++pos == ring_pairs) pos = 0;
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0 && elect_one()) {
      const uint32_t swz = (p.BK == 64) ? SWZ_128B : SWZ_64B;
      const uint32_t pitch = p.BK * 2u, sbo = 8u * pitch;
      const int ksteps = p.BK / 16;
      const uint64_t dbase = make_smem_desc(0, 16, sbo, swz);
      const uint32_t ring16 = smem_u32(s_ring) >> 4, w16 = smem_u32(s_w) >> 4, rowb16 = row_bytes >> 4;
      const uint32_t slot16 = (uint32_t)p.slot_bytes >> 4, pitch16 = pitch >> 4, half16 = half_bytes >> 4, group16 = group_bytes >> 4;
      const uint32_t a_row_full = smem_u32_pinned(row_full), a_row_empty = smem_u32_pinned(row_empty);
      const uint32_t a_tfull = smem_u32_pinned(bar_tfull), a_tempty = smem_u32_pinned(bar_tempty);
      const uint32_t id0 = make_idesc_16(256, 0, 0, 0, p.f16), idu = ((uint32_t)p.Cout >> 3) << 17;   // N field += Cout per row
      const uint32_t nmask = (uint32_t)nacc - 1u, pmask = ((uint32_t)nacc >> 1) - 1u;
      const int pair_sh = nacc_sh - 1;
      const uint64_t dW = dbase + w16;
      const uint32_t C = (uint32_t)p.Cout;
      mbar_wait(&bar_w, 0);
      tc_fence_after();
      // all MMA steps of halo row i of the current strip (`rows` output rows, accumulator of output row 0 = slot j & nmask):
      // output rows [i-1, i+1] clipped to the strip; a row that opens (i+1) starts with accumulate = 0 on the first step
      auto issue_row = [&](int i, int rows, uint32_t j, uint64_t dA) {
        const bool opens = i + 1 < rows;
        const int o_lo = i - 1 < 0 ? 0 : i - 1, o_hi = i + 1 < rows ? i + 1 : rows - 1;
        const uint32_t sa = (j + (uint32_t)o_lo) & nmask;
        const int t0 = o_lo - i + 1;                               // stacked tile of output row o: o - i + 1
        // a span that crosses the end of the accumulator ring is issued as two MMAs
        auto span = [&](int cnt, uint32_t step16, uint32_t wo) {
          if (cnt <= 0) return;
          const int run = cnt < (int)(nacc - sa) ? cnt : (int)(nacc - sa);
          umma2_bf16(tmem_base + sa * C, dA + step16, dW + (wo + st2_region(t0, run) * half16), id0 + run * idu, 1u);
          if (run < cnt)
            umma2_bf16(tmem_base, dA + step16, dW + (wo + st2_region(t0 + run, cnt - run) * half16), id0 + (cnt - run) * idu, 1u);
        };
        bool first = true;
        for (int kc = 0; kc < p.nkc; ++kc)
          for (int dx = 0; dx < 3; ++dx)
            for (int k = 0; k < ksteps; ++k) {
              const uint32_t step16 = kc * slot16 + dx * pitch16 + 2 * k, wo = (uint32_t)(kc * 3 + dx) * group16 + 2 * k;
              if (first) {
                span((opens ? i : o_hi) - o_lo + 1, step16, wo);   // the rows that are already open
                if (opens)
                  umma2_bf16(tmem_base + ((j + (uint32_t)(i + 1)) & nmask) * C, dA + step16, dW + (wo + st2_region(2, 1) * half16),
                             id0 + idu, 0u);
                first = false;
              } else {
                span(o_hi - o_lo + 1, step16, wo);
              }
            }
      };
      int pp = 0; uint32_t fullpar = 0;
      uint32_t j = 0;
      long long u = u_begin;
      asm volatile(".reg .pred p2_rf, p2_te;");                 // split-phase poll results (see the single-CTA folded loop)
#ifdef DCB_STRIP_TIMING
      unsigned long long dbg_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      const long long dbg_t0 = clock64();
#endif
      for (int n, h0, rows, w0; next_strip(u, n, h0, rows, w0);) {
        const int half = rows >> 1;
        bool pre = false, pre_te = false;
        for (int m = 0; m <= half; ++m) {                         // input (halo) rows h0 + 2m - 1 and h0 + 2m
          const uint32_t jp = (j >> 1) + (uint32_t)m;             // running index of the output pair P(m)
          ST_T(c0);
          ST_DECL(c1);
          {
            uint32_t ok_rf = 0, ok_te = 0;
            if (pre) {
              asm volatile("selp.u32 %0, 1, 0, p2_rf;" : "=r"(ok_rf));
              if (pre_te) asm volatile("selp.u32 %0, 1, 0, p2_te;" : "=r"(ok_te));
            }
            if (!ok_rf) mbar_wait_a(a_row_full + 8u * pp, (fullpar >> pp) & 1u);
            fullpar ^= 1u << pp;
            ST_SET(c1); ST_ACC(0, c0, c1);
            if (m < half && !ok_te) mbar_wait_a(a_tempty + 8u * (jp & pmask), ((jp >> pair_sh) & 1u) ^ 1u);
          }
          tc_fence_after();
          ST_T(c2); ST_ACC(1, c1, c2);
          pre = m < half;
          pre_te = m + 1 < half;
          if (pre) {                                              // polls of pair m+1, consumed at the top of the next iteration
            const int ppn = (pp + 1 == ring_pairs) ? 0 : pp + 1;
            asm volatile("mbarrier.test_wait.parity.shared::cta.b64 p2_rf, [%0], %1;" ::"r"(a_row_full + 8u * ppn),
                         "r"((fullpar >> ppn) & 1u) : "memory");
            if (pre_te)
              asm volatile("mbarrier.test_wait.parity.shared::cta.b64 p2_te, [%0], %1;" ::"r"(a_tempty + 8u * ((jp + 1u) & pmask)),
                           "r"((((jp + 1u) >> pair_sh) & 1u) ^ 1u) : "memory");
          }
          const uint64_t dA0 = dbase + (ring16 + (uint32_t)pp * 2u * rowb16), dA1 = dA0 + rowb16;
          if (m >= 1 && m < half && (jp & pmask) != 0u) {        // interior pair, its four accumulators are contiguous
            const uint32_t d0 = tmem_base + (((jp - 1u) & pmask) * 2u) * C;
            if (ksteps == 4) {
              fold2_issue_fast<4>(d0, d0 + 2u * C, dA0, dW, id0 + idu, id0 + 2u * idu, id0 + 3u * idu, p.nkc, slot16, pitch16, half16, group16);
              fold2_issue_fast<4>(d0 + C, d0 + 3u * C, dA1, dW, id0 + idu, id0 + 2u * idu, id0 + 3u * idu, p.nkc, slot16, pitch16, half16, group16);
            } else {
              fold2_issue_fast<2>(d0, d0 + 2u * C, dA0, dW, id0 + idu, id0 + 2u * idu, id0 + 3u * idu, p.nkc, slot16, pitch16, half16, group16);
              fold2_issue_fast<2>(d0 + C, d0 + 3u * C, dA1, dW, id0 + idu, id0 + 2u * idu, id0 + 3u * idu, p.nkc, slot16, pitch16, half16, group16);
            }
          } else {
            issue_row(2 * m - 1, rows, j, dA0);
            issue_row(2 * m, rows, j, dA1);
          }
          ST_T(c3); ST_ACC(2, c2, c3);
          umma2_commit_both(a_row_empty + 8u * pp);
          if (m >= 1) umma2_commit_both(a_tfull + 8u * ((jp - 1u) & pmask));   // output pair P(m-1) is complete
          ST_T(c4); ST_ACC(3, c3, c4); ST_ACC(4, c0, c4);
#ifdef DCB_STRIP_TIMING
          dbg_acc[5] += 1;
#endif
          if (++pp == ring_pairs) pp = 0;
        }
        j += (uint32_t)rows;
      }
#ifdef DCB_STRIP_TIMING
      dbg_acc[6] = (unsigned long long)(clock64() - dbg_t0);
      for (int q = 0; q < 8; ++q) g_strip_dbg[(blockIdx.x >> 1) * 8 + q] = dbg_acc[q];
#endif
    }
  } else {
    const int quarter = warp & 3;
    const int eset = (warp - 2) >> 2;
    const int m = quarter * 32 + lane;
    const float head_b = (FUSED && p.head_kernel) ? (p.head_bias[1] - p.head_bias[0]) : 0.f;
    const uint32_t l_tempty = mapa_u32(smem_u32(bar_tempty), 0);
    const uint32_t t_lane = tmem_base + ((uint32_t)(quarter * 32) << 16);
    const uint32_t pmask = ((uint32_t)nacc >> 1) - 1u;
    uint32_t j = 0;
    long long u = u_begin;
    for (int n, h0, rows, w0; next_strip(u, n, h0, rows, w0);) {
      for (int t = 0; t < rows; t += 2, j += 2) {
        const uint32_t jp = j >> 1;
        if ((int)(jp & 1u) != eset) continue;
        const uint32_t ta = t_lane + (j & (uint32_t)(nacc - 1)) * (uint32_t)p.Cout, tb = ta + (uint32_t)p.Cout;
        const int bar_i = (int)(jp & pmask);
        mbar_wait(&bar_tfull[bar_i], (j >> nacc_sh) & 1u);
        tc_fence_after();
        strip_drain_pair<FUSED>(p, ta, tb, n, h0 + t, w0 + m, s_scale, s_shift, s_wd, head_b, lane, p.n0);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(l_tempty + 8u * bar_i);
      }
    }
  }
  tc_fence_before();
  cluster_sync_all();          // the peer may still signal this CTA's barriers / read its shared memory until here
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// ====================================================================================== flat halo-tile kernel
// conv3x3 for NARROW images (W <= 64: every level below full resolution of a 128^2 training crop, the deep
// levels of a 512^2 image), where a 128-pixel row segment does not exist and the generic kernel re-loads every
// activation tile nine times (once per tap) through L2.
//   * The image is viewed with a one-pixel zero border per row: padded width Wp = W + 2, flattened position
//     f = y * Wp + (x + 1).  In that view EVERY tap is a constant offset: tap (dy, dx) of position f is position
//     f + dy * Wp + dx.  A work item is NT consecutive positions of one image x 128 output channels.
//   * Per 64-channel chunk of K the producer loads ONE pixel buffer - R whole image rows as a single TMA box
//     [64 ch x Wp px x R rows] starting at x = -1, so the zero border (and the rows above / below the image) come
//     from the TMA out-of-bounds fill - and the nine taps are nine row-shifted descriptors into it (the swizzle is a
//     function of the absolute shared-memory address, profiles/r1_umma_row_shift_probe.log).
//   * Swapped orientation: the 128 output channels are the MMA M rows (weights = A operand, streamed in groups of
//     three taps: 3 x [128 x 64] per barrier), the NT positions are the MMA N columns (B operand), so every MMA is
//     N = NT = 192..256 wide and one barrier wait / commit is amortised over 12 MMAs.
//   * Border positions (x = -1, x = W) are computed and thrown away by the epilogue (2 / Wp of the work).
struct TcFlatParams {
  int N, H, W, Wp;
  int C0, C1, nkc;          // K chunks of 64 channels over both sources
  int Cout, mtiles;         // output channels, ceil(Cout / 128)
  int NT, ptiles;           // positions per tile, tiles per image
  int R;                    // image rows per pixel buffer
  int wrows;                // rows of the weight box = min(Cout, 128)
  uint32_t pbuf_bytes;      // R * Wp * 128 rounded up to 1024
  int relu, out_f32;
  int f16;                  // 16-bit element format: 0 = bf16, 1 = fp16
  void* out;
  const float* scale;
  const float* shift;
  int stile;                // bytes of one epilogue warp's transpose tile: 2048 (16-bit outputs) or 4096 (fp32)
  long long* stat_sums;     // STATS instantiation (training forward), see stats_epilogue.cuh
};
constexpr int FL_QUARTETS = 2;                              // epilogue quartets: quartet q drains accumulator stage q (every other item)
constexpr int FL_THREADS = 64 + FL_QUARTETS * 4 * 32;
constexpr uint32_t FL_WSLOT = 3u * 128u * 128u;   // three [128 x 64] bf16 weight tiles

template <bool STATS>
__global__ void __launch_bounds__(FL_THREADS, 1)
tapgemm_tc_flat_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
                       const __grid_constant__ CUtensorMap mapB, const TcFlatParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ uint64_t pb_full[2], pb_empty[2], w_full[2], w_empty[2], bar_tfull[2], bar_tempty[2];
  __shared__ uint32_t tmem_base_smem;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) pdl_trigger();
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* s_pb = smem;                                   // 2 pixel buffers
  uint8_t* s_w = s_pb + 2u * p.pbuf_bytes;                // 2 weight slots
  uint8_t* s_stage = s_w + 2u * FL_WSLOT;                 // one 4 KB transpose tile per epilogue warp
  const int K = p.C0 + p.C1;
  const int num_items = p.N * p.ptiles * p.mtiles;
  uint32_t tmem_cols = 32;
  while (tmem_cols < 2u * (uint32_t)p.NT) tmem_cols <<= 1;
  float st_s = 0.f, st_q = 0.f;                             // STATS: sums of this thread's output channel

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapA0);
    if (p.C1 > 0) tma_prefetch_desc(&mapA1);
    tma_prefetch_desc(&mapB);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&pb_full[i], 1); mbar_init(&pb_empty[i], 1); mbar_init(&w_full[i], 1); mbar_init(&w_empty[i], 1);
      mbar_init(&bar_tfull[i], 1); mbar_init(&bar_tempty[i], 4);
    }
    mbar_fence_init();
  }
  if (warp == 1) { tmem_alloc(&tmem_base_smem, tmem_cols); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;

  // item -> (image, position tile, channel tile); channel tiles of one position tile are neighbours (pixels stay in L2)
  auto decode = [&](int item, int& n, int& f0, int& mt, int& y_lo) {
    mt = item % p.mtiles; item /= p.mtiles;
    const int pt = item % p.ptiles; n = item / p.ptiles;
    f0 = pt * p.NT;
    const int a = f0 - p.Wp - 1;                          // lowest position any tap of the tile reads (may be < 0)
    y_lo = a >= 0 ? a / p.Wp : -((-a + p.Wp - 1) / p.Wp);
  };

  if (warp == 0) {
    if (elect_one()) {
      const int kc0 = p.C0 / 64;
      int pb = 0, ws = 0; uint32_t pb_par = 0, ws_par = 0;   // parities of the NEXT use of each slot's empty barrier
      pdl_wait();                                            // the activations come from the previous kernel of the stream
      for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
        int n, f0, mt, y_lo;
        decode(item, n, f0, mt, y_lo);
        for (int kc = 0; kc < p.nkc; ++kc) {
          const bool second = kc >= kc0;
          const int cc = (second ? kc - kc0 : kc) * 64;
          mbar_wait(&pb_empty[pb], ((pb_par >> pb) & 1u) ^ 1u);
          pb_par ^= 1u << pb;
          mbar_arrive_expect_tx(&pb_full[pb], (uint32_t)p.R * p.Wp * 128u);
          tma_load_4d(second ? &mapA1 : &mapA0, &pb_full[pb], s_pb + (size_t)pb * p.pbuf_bytes, cc, -1, y_lo, n);
          pb ^= 1;
          for (int g = 0; g < 3; ++g) {
            mbar_wait(&w_empty[ws], ((ws_par >> ws) & 1u) ^ 1u);
            ws_par ^= 1u << ws;
            mbar_arrive_expect_tx(&w_full[ws], 3u * (uint32_t)p.wrows * 128u);
            for (int t = 0; t < 3; ++t)
              tma_load_2d(&mapB, &w_full[ws], s_w + (size_t)ws * FL_WSLOT + (size_t)t * 16384u, (g * 3 + t) * K + kc * 64, mt * 128);
            ws ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      const uint32_t idesc = make_idesc_16(128, p.NT, 0, 0, p.f16);
      const uint64_t dbase = make_smem_desc(0, 16, 1024, SWZ_128B);
      const uint32_t pb16 = smem_u32(s_pb) >> 4, w16 = smem_u32(s_w) >> 4, pbuf16 = p.pbuf_bytes >> 4;
      int pb = 0, ws = 0; uint32_t pb_par = 0, ws_par = 0;
      uint32_t it = 0;
      for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
        int n, f0, mt, y_lo;
        decode(item, n, f0, mt, y_lo);
        const uint32_t acc = it & 1u;
        mbar_wait(&bar_tempty[acc], ((it >> 1) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * (uint32_t)p.NT;
        const int base_row = f0 - y_lo * p.Wp;             // buffer row of the tile's first position (>= Wp + 1)
        uint32_t accf = 0;
        for (int kc = 0; kc < p.nkc; ++kc) {
          mbar_wait(&pb_full[pb], (pb_par >> pb) & 1u);
          pb_par ^= 1u << pb;
          const uint32_t prow16 = pb16 + (uint32_t)pb * pbuf16 + (uint32_t)base_row * 8u;   // 128-byte rows = 8 x 16 B
          for (int g = 0; g < 3; ++g) {
            mbar_wait(&w_full[ws], (ws_par >> ws) & 1u);
            ws_par ^= 1u << ws;
            tc_fence_after();
            const int dyo = (g - 1) * p.Wp;                // taps g*3 .. g*3+2 share dy = g - 1
#pragma unroll
            for (int t = 0; t < 3; ++t) {
              const uint64_t da = dbase + (w16 + (uint32_t)ws * (FL_WSLOT >> 4) + (uint32_t)t * 1024u);
              const uint64_t db = dbase + (uint32_t)((int)prow16 + (dyo + t - 1) * 8);
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                umma_bf16(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, accf);
                accf = 1u;
              }
            }
            umma_commit(&w_empty[ws]);
            ws ^= 1;
          }
          umma_commit(&pb_empty[pb]);
          pb ^= 1;
        }
        umma_commit(&bar_tfull[acc]);
      }
    }
  } else {
    // Draining a [128 ch x NT] accumulator through the per-warp transpose tiles takes one quartet longer than the MMAs of
    // a 64 .. 128-channel K take (the statistics experiment: +70 % epilogue work = +70 % kernel time), so two quartets
    // alternate: quartet q owns accumulator stage q.
    const int quarter = warp & 3, eset = (warp - 2) >> 2;
    uint32_t it = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
      if ((int)(it & 1u) != eset) continue;
      int n, f0, mt, y_lo;
      decode(item, n, f0, mt, y_lo);
      const uint32_t acc = it & 1u;
      const int ch0 = mt * 128 + quarter * 32;             // first output channel of this warp
      const bool warp_valid = ch0 < p.Cout;
      const float sc = (warp_valid && p.scale) ? p.scale[ch0 + lane] : 1.f, sh = (warp_valid && p.shift) ? p.shift[ch0 + lane] : 0.f;
      auto pix_index = [&](int mm) -> long long {
        const int f = f0 + mm, y = f / p.Wp, xp = f - y * p.Wp;
        if (y >= p.H || xp < 1 || xp > p.W) return -1;
        return (long long)((((size_t)n * p.H + y) * p.W + (xp - 1)) * p.Cout + ch0);
      };
      mbar_wait(&bar_tfull[acc], (it >> 1) & 1u);
      tc_fence_after();
      epilogue_swapped<STATS>(tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * (uint32_t)p.NT, p.NT, warp_valid, sc, sh, p.relu,
                              p.out_f32, p.out, s_stage + (eset * 4 + quarter) * p.stile, lane, pix_index, p.f16, &st_s, &st_q);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_tempty[acc]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) { tc_fence_after(); tmem_dealloc(tmem_base, tmem_cols); }
  if constexpr (STATS) {
    // the grid is a multiple of mtiles, so every item of this CTA has the same channel tile mt; the four epilogue warps
    // of a quartet own 32 channels each: written as four accumulator blocks per quartet (layout of stats_cta_finish)
    float* dump = reinterpret_cast<float*>(s_pb);
    if (warp >= 2) {
      const int quarter = warp & 3, eset = (warp - 2) >> 2;
      float* d = dump + ((size_t)((eset * 4 + quarter) * 16) + (lane >> 1)) * 4 + (lane & 1);
      d[0] = st_s; d[2] = st_q;
    }
    __syncthreads();
    const int mt = blockIdx.x % p.mtiles;
    stats_cta_finish(dump, FL_QUARTETS, 4, [&](int bi) { return mt * 128 + bi * 32; }, p.Cout, p.stat_sums);
  }
}

// ---------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(sym);
  });
  return fn;
}

// 16-bit tensor map (f16: fp16 elements, else bf16); dims/strides innermost first; strides[i] is the byte stride of dim i+1
static int make_map(CUtensorMap* out, int f16, const void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                    const uint32_t* box, int swizzle_bytes) {
  typedef std::tuple<const void*, int, std::vector<uint64_t>, std::vector<uint64_t>, std::vector<uint32_t>, int, int> Key;
  static std::map<Key, CUtensorMap> cache;
  static std::mutex mu;
  Key key(ptr, rank, std::vector<uint64_t>(dims, dims + rank), std::vector<uint64_t>(strides_bytes, strides_bytes + rank - 1),
          std::vector<uint32_t>(box, box + rank), swizzle_bytes, f16);
  std::lock_guard<std::mutex> lock(mu);
  auto it = cache.find(key);
  if (it != cache.end()) { *out = it->second; return DCB_OK; }
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return fail(DCB_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available from the driver");
  cuuint64_t gdim[5]; cuuint64_t gstr[4]; cuuint32_t bx[5]; cuuint32_t es[5];
  for (int i = 0; i < rank; ++i) { gdim[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
  for (int i = 0; i < rank - 1; ++i) gstr[i] = strides_bytes[i];
  CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                          : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = enc(out, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(ptr), gdim, gstr, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    return fail(DCB_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d): rank %d dims [%llu,%llu,%llu,..] box [%u,%u,%u,..] swizzle %d",
                (int)r, rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
                (unsigned long long)(rank > 2 ? dims[2] : 0), box[0], rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0,
                swizzle_bytes);
  }
  if (cache.size() > 4096) cache.clear();
  cache[key] = *out;
  return DCB_OK;
}

// The four views the kernels read and write.  `pitch` is the channel stride of a pixel (>= C: a channel slice of a
// wider tensor).
// NHWC tensor [N][H][W][C], boxes of {bc channels, bw columns, bh rows, bn images}
static int map_nhwc(CUtensorMap* m, int f16, const void* ptr, int N, int H, int W, int C, int pitch, uint32_t bc, uint32_t bw,
                    uint32_t bh, uint32_t bn, int swz) {
  const uint64_t dims[4] = {(uint64_t)C, (uint64_t)W, (uint64_t)H, (uint64_t)N};
  const uint64_t str[3] = {(uint64_t)pitch * 2, (uint64_t)W * pitch * 2, (uint64_t)H * W * pitch * 2};
  const uint32_t box[4] = {bc, bw, bh, bn};
  return make_map(m, f16, ptr, 4, dims, str, box, swz);
}
// NHWC tensor with the image and row axes merged: [rows = N*H][W][C], boxes of {bc, bw, bh rows}
static int map_rows(CUtensorMap* m, int f16, const void* ptr, long long rows, int W, int C, uint32_t bc, uint32_t bw, uint32_t bh,
                    int swz) {
  const uint64_t dims[3] = {(uint64_t)C, (uint64_t)W, (uint64_t)rows};
  const uint64_t str[2] = {(uint64_t)C * 2, (uint64_t)W * C * 2};
  const uint32_t box[3] = {bc, bw, bh};
  return make_map(m, f16, ptr, 3, dims, str, box, swz);
}
// sub-pixel view of a [N][2h][2w][C] tensor: [rows = N*h][a = 2][w][b = 2][C] -> innermost first {C, b, w, a, rows};
// boxes of {bc, 1, bw, 1, bh}: bw pixels of one (a, b) sub-position in each of bh rows
static int map_subpixel(CUtensorMap* m, int f16, const void* ptr, long long rows, int w, int C, int pitch, uint32_t bc, uint32_t bw,
                        uint32_t bh, int swz) {
  const uint64_t dims[5] = {(uint64_t)C, 2, (uint64_t)w, 2, (uint64_t)rows};
  const uint64_t str[4] = {(uint64_t)pitch * 2, (uint64_t)2 * pitch * 2, (uint64_t)2 * w * pitch * 2, (uint64_t)4 * w * pitch * 2};
  const uint32_t box[5] = {bc, 1, bw, 1, bh};
  return make_map(m, f16, ptr, 5, dims, str, box, swz);
}
// weight matrix [rows][K], boxes of {bk, brows}
static int map_weights(CUtensorMap* m, int f16, const void* ptr, int K, int rows, uint32_t bk, uint32_t brows, int swz) {
  const uint64_t dims[2] = {(uint64_t)K, (uint64_t)rows};
  const uint64_t str[1] = {(uint64_t)K * 2};
  const uint32_t box[2] = {bk, brows};
  return make_map(m, f16, ptr, 2, dims, str, box, swz);
}

static int pick_pow2_box(int extent, int maxbox) {
  // power-of-two box <= maxbox covering `extent` with the least padding (ties -> larger box);
  // boxes below 8 are only used when the extent itself is smaller
  int lo = 1;
  while (lo < 8 && lo < extent) lo <<= 1;
  if (lo > maxbox) lo = maxbox;
  int best = lo; double best_waste = 1e30;
  for (int b = lo; b <= maxbox; b <<= 1) {
    int tiles = (extent + b - 1) / b;
    double waste = (double)tiles * b / extent;
    if (waste <= best_waste + 1e-9) { best_waste = waste; best = b; }
  }
  return best;
}

// swapped orientation policy: DCB_POLICY_SWAP_MIN_COUT = smallest Cout for which the swapped orientation is used
// (<= 128 always required); 0 disables.  Default chosen from per-layer measurements (profiles/).
static int swap_min_cout() { return policy(DCB_POLICY_SWAP_MIN_COUT); }
static bool swap_allowed(int Nout) { return swap_min_cout() > 0 && Nout >= swap_min_cout() && Nout <= 128; }

// maximum dynamic shared memory of each kernel family (cudaFuncAttributeMaxDynamicSharedMemorySize)
constexpr int TC_SMEM_MAX = 206 * 1024, ST_SMEM_MAX = 224 * 1024, FL_SMEM_MAX = 224 * 1024;

// strip kernel plan for a launch that computes Nsub of the layer's Nout output channels (Nsub < Nout: the layer is
// run as Nout / Nsub launches because the weights of all channels do not fit next to a useful halo ring);
// returns false when the layer is not eligible
static bool plan_strip(const TapGeom& g, int C0, int C1, int Nout, int Nsub, bool fused, TcStripParams& p, size_t& dyn_smem,
                       bool stats = false) {
  if (!policy(DCB_POLICY_STRIP)) return false;
  // batch statistics in the epilogue: folded single-CTA launches over all output channels only; 8 x 2 KB of scratch
  // tiles behind the ring (where the swapped orientation keeps its transpose tiles)
  if (stats && (fused || Nsub != Nout || Nout > 64)) return false;
  if (g.ntaps != 9 || g.zsub > 1 || g.sy != 1) return false;
  if (g.GW % 128 != 0 || Nsub > 128 || Nsub % 32 != 0 || Nout % Nsub != 0) return false;
  const int K = C0 + C1;
  const int BK = (C0 % 64 == 0 && C1 % 64 == 0) ? 64 : 32;
  const int nkc = K / BK;
  const size_t w_bytes = ((size_t)9 * K * Nsub * 2 + 1023) & ~(size_t)1023;
  // dynamic shared memory: 224 KB minus the 1 KB alignment slack; the swapped epilogue also needs 4 x 4 KB there
  const size_t budget_all = 223 * 1024, stage_tiles = 4 * 4096;
  // swapped orientation (256-pixel segments, N = 256 per MMA) whenever the image is wide enough
  // the fused head / pool epilogues exist for the normal orientation only
  // Cout = 64 is faster folded (13 MMAs of N = 192 per 128 pixels) than swapped (36 MMAs of N = 256 per 256 pixels with
  // half of the 128 M rows empty): measured 0.050/0.056 -> 0.042/0.046 ms on the 256^2 layers; swapped strips are
  // for Cout = 128 only
  const bool no_fold_pref = !policy(DCB_POLICY_FOLD);
  int swap = (!fused && !stats && swap_allowed(Nsub) && g.GW % 256 == 0 && (Nsub > 64 || no_fold_pref || g.GH % 2 != 0)) ? 1 : 0;
  int slot = 0, ring = 0;
  for (; swap >= 0; --swap) {
    const int px = swap ? 256 : 128;
    const size_t budget = budget_all - ((swap || stats) ? stage_tiles : 0);
    slot = ((px + 2) * BK * 2 + 1023) & ~1023;
    // the MMA reads 128 weight rows starting at each (tap, kc) block: keep those reads inside the allocation
    if (w_bytes + (size_t)4 * nkc * slot <= budget) { ring = (int)((budget - w_bytes) / ((size_t)nkc * slot)); break; }
  }
  if (swap < 0) return false;
  if (ring > ST_MAX_RING) ring = ST_MAX_RING;
  memset(&p, 0, sizeof(p));
  p.N = g.N; p.H = g.GH; p.W = g.GW; p.C0 = C0; p.C1 = C1; p.BK = BK; p.nkc = nkc; p.Cout = Nsub; p.OC = Nout;
  p.ring = ring; p.slot_bytes = slot; p.swap = swap; p.wsegs = g.GW / (swap ? 256 : 128);
  const bool no_fold = !policy(DCB_POLICY_FOLD);
  p.fold = (!swap && !no_fold && (Nsub == 32 || Nsub == 64) && g.GH % 2 == 0 && ring >= 4) ? 1 : 0;
  if (fused && (g.GH % 2 != 0)) return false;          // row pairs of the fused pool must not straddle strips
  if (Nsub < Nout && !p.fold) return false;            // channel-split launches only pay with the folded issue
  if (stats && !p.fold) return false;
  p.gran = (g.GH % 2 == 0) ? 2 : 1;
  dyn_smem = w_bytes + (size_t)ring * nkc * slot + ((swap || stats) ? stage_tiles : 0) + 1024;
  return true;
}

struct FlatPlan { TcFlatParams p; size_t dyn; int grid; bool stats; };

// flat halo-tile kernel plan; false when the layer is not eligible
static bool plan_flat(const TapGeom& g, int C0, int C1, int Nout, int out_f32, bool stats, FlatPlan& fp) {
  const int flat_policy = policy(DCB_POLICY_FLAT);
  if (flat_policy == 0 || g.ntaps != 9 || g.zsub > 1 || g.sy != 1) return false;
  if (C0 % 64 != 0 || C1 % 64 != 0 || Nout < 64 || g.GW > 64 || g.GW < 16) return false;
  const int Wp = g.GW + 2;
  const long long positions = (long long)g.GH * Wp;
  if (positions < 512) return false;     // tiny maps: too much of a 192..256-position tile would be padding
  TcFlatParams& p = fp.p;
  memset(&p, 0, sizeof(p));
  const size_t stile = out_f32 ? 4096 : 2048;            // per-warp transpose tile of the epilogue
  const size_t budget = 223 * 1024 - 2 * (size_t)FL_WSLOT - FL_QUARTETS * 4 * stile;
  int NT = 0, R = 0; uint32_t pbuf = 0;
  for (int cand : {256, 192, 128}) {
    R = (cand + 3 * Wp + 1 + Wp - 1) / Wp;
    pbuf = ((uint32_t)R * Wp * 128u + 1023u) & ~1023u;
    if (R <= 256 && 2 * (size_t)pbuf <= budget) { NT = cand; break; }
  }
  if (!NT) return false;
  // Measured (scripts/one_layer.py, profiles/r1_flat_kernel_ab.txt): the coarse work items (NT positions x 128 channels x all
  // of K) only pay when every SM gets several of them; otherwise the generic kernel's finer tiles balance better.
  {
    const bool force = flat_policy >= 2;
    const long long items = (long long)g.N * ((positions + NT - 1) / NT) * cdiv(Nout, 128);
    if (!force && items < 4LL * sm_count()) return false;
  }
  p.N = g.N; p.H = g.GH; p.W = g.GW; p.Wp = Wp; p.C0 = C0; p.C1 = C1; p.nkc = (C0 + C1) / 64;
  p.Cout = Nout; p.mtiles = cdiv(Nout, 128); p.NT = NT; p.ptiles = (int)((positions + NT - 1) / NT); p.R = R;
  p.wrows = Nout < 128 ? Nout : 128; p.pbuf_bytes = pbuf; p.stile = (int)stile;
  p.out_f32 = out_f32; p.f16 = g.f16;
  fp.dyn = 2 * (size_t)pbuf + 2 * (size_t)FL_WSLOT + FL_QUARTETS * 4 * stile + 1024;
  const int items = p.N * p.ptiles * p.mtiles;
  fp.grid = items < sm_count() ? items : sm_count();
  fp.stats = false;
  // The flat kernel is bound by its four epilogue warps (one 32 x 32 transpose per 32 pixels); the statistics add ~70 % to
  // that loop (measured 28 -> 47 us on the 64 -> 64 layer of a 32 x 64^2 batch, profiles/r2_stats_epilogue_bench.txt) - more
  // than the BatchNorm pass they save.  Only on request (policy fused_bn = 3, the tests).
  if (stats && !out_f32 && policy(DCB_POLICY_FUSED_BN) >= 3) {
    // every CTA keeps one channel tile (its threads accumulate one channel each)
    const int gs = fp.grid - fp.grid % p.mtiles;
    if (gs >= p.mtiles) { fp.grid = gs; fp.stats = true; }
  }
  return true;
}

struct GenericPlan { TcFwdParams p; size_t dyn; int grid; bool pool, stats; };

// generic kernel plan for Nout output channels written with a channel pitch of out_pitch (>= Nout); pool: the 2x2
// max-pooled copy in the epilogue; stats: batch statistics requested.  Returns null, or why the layer is not supported.
static const char* plan_generic(const TapGeom& g, int C0, int C1, int Nout, int out_pitch, int out_f32, bool pool, bool stats,
                                GenericPlan& gp) {
  TcFwdParams& p = gp.p;
  memset(&p, 0, sizeof(p));
  const int ntaps = g.ntaps;
  const bool convT_fwd = g.zsub > 1;
  const bool convT_dgrad = (g.sy == 2);
  p.mode = convT_fwd ? 1 : (convT_dgrad ? 2 : 0);
  p.N = g.N; p.GH = g.GH; p.GW = g.GW;
  p.ntaps = ntaps;
  for (int t = 0; t < ntaps; ++t) { p.dy[t] = g.dy[t]; p.dx[t] = g.dx[t]; }
  p.C0 = C0; p.C1 = C1;
  p.BK = (C0 % 64 == 0 && C1 % 64 == 0) ? 64 : 32;
  p.Cz = Nout;
  p.Ntot = convT_fwd ? 4 * Nout : Nout;
  p.OH = g.OH; p.OW = g.OW; p.OC = out_pitch;
  p.osy = g.osy; p.osx = g.osx; p.ody = g.ody; p.odx = g.odx;
  p.out_f32 = out_f32;
  p.f16 = g.f16;
  // Swapped orientation for narrow outputs: with <= 128 output channels the normal orientation spends the
  // A-operand read time (128 pixel rows per MMA) on an N of 32..128; swapped, every MMA covers 256 pixels.
  {
    const long long px = (long long)g.N * g.GH * g.GW;
    // measured (profiles/r1_layer_ab.txt): pays for conv3x3 with 64..128 output channels, not for the 1-tap convT GEMMs
    // the pooled epilogue is cheaper in the pixels-as-M orientation (two epilogue quartets; profiles/r2_pool_ab.txt)
    p.swap = (p.mode == 0 && !pool && !stats && swap_allowed(Nout) && px / 256 * cdiv(p.Ntot, 128) >= sm_count() / 2) ? 1 : 0;
  }
  const int TM = p.swap ? 256 : TC_BM;
  // ---- M tiling
  if (p.mode == 0) {
    p.bw = pick_pow2_box(g.GW, TM);
    // the pooled epilogue needs whole 2x2 windows inside a tile: rows wide enough for a one-row tile are split in two
    if (pool && p.bw == TM && TM >= 4) p.bw = TM / 2;
    p.bh = pick_pow2_box(g.GH, TM / p.bw);
    p.bn = TM / (p.bw * p.bh);
    p.tiles_w = cdiv(g.GW, p.bw); p.tiles_h = cdiv(g.GH, p.bh); p.tiles_n = cdiv(g.N, p.bn);
  } else {
    p.bw = pick_pow2_box(g.GW, TM);
    p.bh = TM / p.bw; p.bn = 1;
    p.tiles_w = cdiv(g.GW, p.bw); p.tiles_h = cdiv((long long)g.N * g.GH, p.bh); p.tiles_n = 1;
  }
  const int num_mtiles = p.tiles_w * p.tiles_h * p.tiles_n;
  // pooled epilogue: conv3x3 only, 16-bit outputs, whole 2x2 windows inside every tile
  if (pool && (p.mode != 0 || out_f32 || (g.GH & 1) || (g.GW & 1) || (p.bw & 1) || (p.bh & 1) || (p.swap && p.bw % 32 != 0) ||
               out_pitch != Nout))
    return "fused max-pool not available for this layer shape";
  gp.pool = pool;
  // ---- N tiling: largest tile that still gives every SM work
  // an N tile may span several convT sub-positions (the epilogue resolves them per 32-column block)
  // Cost model from the issue-rate probes (profiles/r1_umma_rate_probe.log): one M=128 MMA occupies the tensor pipe for
  // ~89 cycles whatever N <= 128 is, and for 128 cycles at N = 256, so a tile costs (MMAs per tile) x c(BN) and the launch
  // costs waves x that.  Halving BN below 128 never shortens a tile; it only pays when it removes a wave.
  int BN = 32;
  {
    double best = 1e30;
    for (int cand : {256, 192, 128, 96, 64, 32}) {
      if (cand > p.Ntot || p.Ntot % cand != 0) continue;
      const long long tiles = (long long)num_mtiles * (p.Ntot / cand);
      const long long waves = (tiles + sm_count() - 1) / sm_count();
      const double cost = (double)waves * (cand <= 128 ? 89.0 : 89.0 + (cand - 128) * (39.0 / 128.0));
      if (cost < best - 1e-9) { best = cost; BN = cand; }     // ties: the larger tile (fewer activation re-loads)
    }
  }
  if (p.swap) BN = p.Ntot < 128 ? p.Ntot : 128;       // rows of the weight TMA box
  p.BN = BN;
  const size_t stage_bytes = (size_t)TM * p.BK * 2 + (size_t)(p.swap ? 128 : BN) * p.BK * 2;
  // 16-bit outputs of the convT forward leave through TMA stores (two 8 KB staging tiles per epilogue quartet): its
  // scattered 64-byte runs saturate the LSU pipe as plain stores (profiles/r2_convT_ncu.txt).  The conv3x3 layers on this
  // kernel are operand-traffic bound and lose more from the smaller stage ring than the stores gain (measured; policy 2
  // = TMA stores there too).
  const bool with_stats = stats && !pool && !out_f32 && p.mode != 2 && out_pitch == Nout;
  p.tma_store = (!p.swap && !out_f32 && !pool && !with_stats && p.mode != 2 &&
                 (policy(DCB_POLICY_TMA_STORE) >= 2 || (policy(DCB_POLICY_TMA_STORE) == 1 && p.mode == 1))) ? 1 : 0;
  const size_t staging = p.tma_store ? 2 * 16384 : 0;
  int stages = (int)((200 * 1024 - staging) / stage_bytes);
  if (stages > TC_MAX_STAGES) stages = TC_MAX_STAGES;
  if (stages < 2) return "tile does not fit shared memory";
  p.stages = stages;
  gp.dyn = stages * stage_bytes + staging + 1024;
  const int num_ntiles = p.swap ? cdiv(p.Ntot, 128) : p.Ntot / BN;
  const int num_tiles = num_mtiles * num_ntiles;
  gp.grid = num_tiles < sm_count() ? num_tiles : sm_count();
  // every CTA keeps ONE N tile (its register accumulators are per 32-column block of the tile): the round-robin
  // schedule tile = blockIdx.x + i * gridDim.x does that when the grid is a multiple of the N-tile count
  const int stats_grid = gp.grid - gp.grid % num_ntiles;
  gp.stats = with_stats && stats_grid >= num_ntiles;
  if (gp.stats) gp.grid = stats_grid;
  return nullptr;
}

// The forward variant of one call and its complete plan (choose_fwd).
struct FwdPlan {
  enum Kind { UNSUPPORTED, GENERIC, FLAT, STRIP, STRIP_CLUSTER, STRIP_PAIR } kind;
  const char* error;        // UNSUPPORTED: why
  bool fused;               // STRIP / STRIP_PAIR: head and / or pool in the epilogue
  bool stats;               // the launch also writes the batch statistics
  int slice;                // GENERIC: output channels per launch (Nout, or 512 for wider outputs)
  GenericPlan gen;          // GENERIC: plan of the first slice
  FlatPlan flat;
  TcStripParams sp;         // STRIP*: parameters of one launch (n0 set per launch)
  size_t strip_dyn;
  int strip_grid;
};

// Which kernel a forward-type call (conv3x3 fwd / dgrad, convT2x2 fwd / dgrad) runs, from the shape, the requested
// epilogue fusions and statistics, and the dispatch policy.  Reads only policy() and sm_count().
static FwdPlan choose_fwd(const TapGeom& g, int C0, int C1, int Nout, const TcFusion* fuse, bool stats, int out_f32) {
  FwdPlan c;
  memset(&c, 0, sizeof(c));
  auto unsupported = [&](const char* why) { c.kind = FwdPlan::UNSUPPORTED; c.error = why; return c; };
  auto generic = [&](int slice, bool pool, bool with_stats) {
    c.kind = FwdPlan::GENERIC; c.slice = slice;
    if (const char* why = plan_generic(g, C0, C1, slice, Nout, out_f32, pool, with_stats, c.gen)) return unsupported(why);
    c.stats = c.gen.stats;
    return c;
  };
  // Small outputs keep the channel-slab BatchNorm kernel, which takes statistics and applies them in ~7 us (2 MB) - less
  // than the one-pass kernel plus the epilogue's extra work (measured gate; policy fused_bn = 3 = wherever available)
  if (stats && policy(DCB_POLICY_FUSED_BN) < 3 &&
      (long long)g.N * g.OH * g.OW * Nout * 2 < (4LL << 20))
    stats = false;
  const bool fused = fuse != nullptr;
  if (Nout > 512) {
    // wide outputs (the dgrad of a 768-channel concat in the 'upsampling' graph): slices of <= 512 channels through the
    // generic kernel, each writing its channel range of the full-pitch output
    if (fused) return unsupported("fused epilogue not available for this layer");
    if (g.zsub > 1) return unsupported("bf16 convT with more than 512 output channels is not built");
    return generic(512, false, false);
  }
  if (fused && out_f32) return unsupported("fused epilogue not available for this layer");
  // a pool-only fusion that the strip kernel cannot take (more than 64 output channels, narrow images) goes to the
  // generic kernel's pooled epilogue
  const bool pool_only = fused && fuse->pool_out && !fuse->head_kernel;
  TcStripParams& sp = c.sp;
  const bool strip_stats = stats && plan_strip(g, C0, C1, Nout, Nout, false, sp, c.strip_dyn, true);
  bool strip_ok = strip_stats || (!(fused && fuse->pool_out && Nout > 64) && plan_strip(g, C0, C1, Nout, Nout, fused, sp, c.strip_dyn));
  const bool no_nsplit = !policy(DCB_POLICY_NSPLIT);
  if (!strip_ok && !fused && !no_nsplit && Nout == 64) strip_ok = plan_strip(g, C0, C1, Nout, 32, fused, sp, c.strip_dyn);
  if (fused && !strip_ok) {
    if (pool_only) return generic(Nout, true, false);
    return unsupported("fused epilogue not available for this layer");
  }
  if (strip_ok) {
    c.fused = fused;
    // CTA-pair variant of the folded loop (cta_group::2 MMAs): the stacked weights take 5/3 of the single-CTA footprint
    // per CTA (one region per span shape); used when a ring of at least three row pairs still fits next to them
    if (sp.fold && !strip_stats && policy(DCB_POLICY_PAIR) && (sp.N * sp.wsegs) % 2 == 0 && sp.H % 2 == 0 && sm_count() >= 2) {
      const size_t w2 = ((size_t)15 * sp.nkc * sp.Cout * sp.BK * 2 + 1023) & ~(size_t)1023;
      const size_t budget = 223 * 1024;
      const size_t rowb = (size_t)sp.nkc * sp.slot_bytes;
      int ring2 = w2 < budget ? (int)((budget - w2) / rowb) : 0;
      if (ring2 > ST_MAX_RING) ring2 = ST_MAX_RING;
      ring2 &= ~1;
      if (ring2 >= 6) {
        c.kind = FwdPlan::STRIP_PAIR;
        sp.ring = ring2;
        c.strip_dyn = w2 + (size_t)ring2 * rowb + 1024;
        const long long units2 = (long long)(sp.N * sp.wsegs / 2) * (sp.H / 2);
        c.strip_grid = 2 * (units2 < sm_count() / 2 ? (int)units2 : sm_count() / 2);
        return c;
      }
    }
    const long long units = (long long)sp.N * sp.wsegs * cdiv(sp.H, sp.gran);
    c.kind = FwdPlan::STRIP;
    c.strip_grid = units < sm_count() ? (int)units : sm_count();
    sp.nclu = 1;
    if (strip_stats) { c.stats = true; return c; }
    // channel-split layer (two groups of output channels): ONE launch of two-CTA clusters that share every halo row
    // through TMA multicast instead of two launches that each read the whole input
    if (sp.fold && !fused && Nout == 2 * sp.Cout && sp.nkc % 2 == 0 && policy(DCB_POLICY_NSPLIT) == 1 && sm_count() >= 2) {
      c.kind = FwdPlan::STRIP_CLUSTER;
      sp.nclu = 2;
      c.strip_grid = 2 * (units < sm_count() / 2 ? (int)units : sm_count() / 2);
    }
    return c;
  }
  // A training forward that wants its batch statistics goes to the generic kernel (statistics in the epilogue, +2 us)
  // rather than to the flat kernel (no statistics at the default policy): what the flat kernel gains on the conv (~20 %
  // on 64-pixel rows) is less than the separate statistics pass it would leave to the BatchNorm kernel
  // (scripts/train_time.py flat=0 / 1: 2.589 vs 2.609 ms per step before this rule).
  if (!(stats && policy(DCB_POLICY_FUSED_BN) == 2) && plan_flat(g, C0, C1, Nout, out_f32, stats, c.flat)) {
    c.kind = FwdPlan::FLAT;
    c.stats = c.flat.stats;
    return c;
  }
  return generic(Nout, false, stats);
}

// dcb_last_kernel() name of a planned forward (tests and profiles/ refer to these names)
static const char* fwd_kernel_name(const FwdPlan& c) {
  const TcStripParams& sp = c.sp;
  switch (c.kind) {
    case FwdPlan::GENERIC:
      if (c.stats) return "generic_stats";
      if (c.gen.pool) return c.gen.p.swap ? "generic_swap_pool" : "generic_pool";
      return c.gen.p.swap ? "generic_swap" : "generic";
    case FwdPlan::FLAT: return c.stats ? "flat_stats" : "flat";
    case FwdPlan::STRIP_PAIR: return c.fused ? "strip_pair_fused" : (sp.Cout < sp.OC ? "strip_pair_nsplit" : "strip_pair");
    case FwdPlan::STRIP_CLUSTER: return "strip_fold_nsplit_cluster";
    case FwdPlan::STRIP:
      if (c.stats) return "strip_fold_stats";
      return sp.fold ? (c.fused ? "strip_fold_fused" : (sp.Cout < sp.OC ? "strip_fold_nsplit" : "strip_fold"))
                     : (sp.swap ? "strip_swap" : (c.fused ? "strip_fused" : "strip"));
    default: return "";
  }
}

#ifdef DCB_STRIP_TIMING
static void print_strip_timing(const FwdPlan& c, cudaStream_t st) {
  cudaStreamSynchronize(st);
  if (c.kind == FwdPlan::STRIP_PAIR) {
    const int pairs = c.strip_grid / 2;
    static unsigned long long h[148 * 8];
    cudaMemcpyFromSymbol(h, g_strip_dbg, sizeof(h));
    double a[8] = {0};
    for (int b = 0; b < pairs; ++b) for (int q = 0; q < 8; ++q) a[q] += (double)h[b * 8 + q] / pairs;
    fprintf(stderr, "[strip pair timing] per leader: steps (two halo rows of both CTAs) %.0f | cycles/step: row_full wait %.0f, tempty wait "
            "%.0f, issue %.0f, commit %.0f, total %.0f | loop cycles %.0f\n", a[5], a[0] / a[5], a[1] / a[5], a[2] / a[5], a[3] / a[5],
            a[4] / a[5], a[6]);
    return;
  }
  const int grid = c.strip_grid;
  static unsigned long long h[148 * 8];
  cudaMemcpyFromSymbol(h, g_strip_dbg, sizeof(h));
  double a[8] = {0};
  for (int b = 0; b < grid; ++b) for (int q = 0; q < 8; ++q) a[q] += (double)h[b * 8 + q] / grid;
  static unsigned long long h2[148 * 16];
  cudaMemcpyFromSymbol(h2, g_strip_dbg2, sizeof(h2));
  double e[16] = {0};
  for (int b = 0; b < grid; ++b) for (int q = 0; q < 16; ++q) e[q] += (double)h2[b * 16 + q] / grid;
  fprintf(stderr, "[strip timing] producer: rows %.0f, row_empty wait %.0f cycles/row | epilogue quartet 0: tiles %.0f, tfull wait %.0f, "
          "work %.0f (tmem ld %.0f, math+store %.0f) cycles/tile | quartet 1: tiles %.0f, tfull wait %.0f, work %.0f (ld %.0f, math %.0f)\n",
          e[1], e[0] / e[1], e[3], e[2] / e[3], e[4] / e[3], e[5] / e[3], e[6] / e[3], e[8], e[7] / e[8], e[9] / e[8], e[10] / e[8], e[11] / e[8]);
  fprintf(stderr, "[strip timing] per CTA: fast rows %.0f | cycles/row: row_full wait %.0f, tempty wait %.0f, issue %.0f, commit %.0f, "
          "total %.0f | loop cycles %.0f\n", a[5], a[0] / a[5], a[1] / a[5], a[2] / a[5], a[3] / a[5], a[4] / a[5], a[6]);
}
#endif

// strip kernel launches of a STRIP / STRIP_CLUSTER / STRIP_PAIR plan: one launch per group of output channels
static int launch_strip(const TapGeom& g, FwdPlan& c, const void* s0, int C0, const void* s1, int C1, const void* B, int Nout,
                        void* out, const float* scale, const float* shift, int relu, int out_f32, cudaStream_t st,
                        const TcFusion* fuse, TcStats* stats) {
  TcStripParams& sp = c.sp;
  sp.relu = relu; sp.out_f32 = out_f32; sp.out = reinterpret_cast<__nv_bfloat16*>(out); sp.scale = scale; sp.shift = shift;
  sp.f16 = g.f16;
  sp.need_y = 1;
  if (c.fused) {
    sp.head_kernel = fuse->head_kernel; sp.head_bias = fuse->head_bias; sp.logit = fuse->logit; sp.prob = fuse->prob;
    sp.need_y = fuse->need_y; sp.pool_out = reinterpret_cast<__nv_bfloat16*>(fuse->pool_out);
  }
  if (c.stats) sp.stat_sums = stats->sums;
  const bool pair = c.kind == FwdPlan::STRIP_PAIR;
  CUtensorMap mA0, mA1, mT0{}, mT1{}, mB;
  const int swz = sp.BK * 2;
  const uint32_t mainw = sp.swap ? 256u : 130u;
  if (int e = map_nhwc(&mA0, g.f16, s0, g.N, g.IH, g.IW, C0, C0, sp.BK, mainw, 1, 1, swz)) return e;
  if (!pair) { if (int e = map_nhwc(&mT0, g.f16, s0, g.N, g.IH, g.IW, C0, C0, sp.BK, 2, 1, 1, swz)) return e; }
  if (C1 > 0) {
    if (int e = map_nhwc(&mA1, g.f16, s1, g.N, g.IH, g.IW, C1, C1, sp.BK, mainw, 1, 1, swz)) return e;
    if (!pair) { if (int e = map_nhwc(&mT1, g.f16, s1, g.N, g.IH, g.IW, C1, C1, sp.BK, 2, 1, 1, swz)) return e; }
  } else { mA1 = mA0; mT1 = mT0; }
  // the pair kernel's CTAs each load half of the weight rows of a launch
  if (int e = map_weights(&mB, g.f16, B, 9 * (C0 + C1), Nout, sp.BK, pair ? sp.Cout / 2 : sp.Cout, swz)) return e;
  const bool pdl = policy(DCB_POLICY_PDL) != 0;
  const int per_launch = c.kind == FwdPlan::STRIP_CLUSTER ? Nout : sp.Cout;   // output channels of one launch
  for (sp.n0 = 0; sp.n0 < Nout; sp.n0 += per_launch) {
    int e;
    if (pair) {
      e = launch(c.fused ? tapgemm_tc_strip2_kernel<true> : tapgemm_tc_strip2_kernel<false>, "tapgemm_tc_strip2_kernel", c.strip_grid,
                 ST_THREADS, c.strip_dyn, ST_SMEM_MAX, st, pdl, 2, mA0, mA1, mB, sp);
    } else {
      auto* k = c.stats ? tapgemm_tc_strip_kernel<false, true, true>
                : c.fused ? (sp.fold ? tapgemm_tc_strip_kernel<true, true> : tapgemm_tc_strip_kernel<true, false>)
                          : (sp.fold ? tapgemm_tc_strip_kernel<false, true> : tapgemm_tc_strip_kernel<false, false>);
      e = launch(k, "tapgemm_tc_strip_kernel", c.strip_grid, ST_THREADS, c.strip_dyn, ST_SMEM_MAX, st, pdl,
                 c.kind == FwdPlan::STRIP_CLUSTER ? 2 : 0, mA0, mA1, mT0, mT1, mB, sp);
    }
    if (e) return e;
  }
#ifdef DCB_STRIP_TIMING
  if ((pair || (c.kind == FwdPlan::STRIP && !c.stats && sp.fold)) && getenv("DCB_STRIP_TIMING_PRINT")) print_strip_timing(c, st);
#endif
  return DCB_OK;
}

// generic kernel launches of a GENERIC plan: one per slice of c.slice output channels (a narrower last slice is planned
// here, so c.gen ends as the plan of the last launch)
static int launch_generic(const TapGeom& g, FwdPlan& c, const void* s0, int C0, const void* s1, int C1, const void* B, int Nout,
                          void* out, const float* scale, const float* shift, int relu, int out_f32, cudaStream_t st,
                          const TcFusion* fuse, TcStats* stats) {
  const size_t esz = out_f32 ? 4 : 2;
  const size_t wrow = (size_t)g.ntaps * (C0 + C1);
  for (int n0 = 0; n0 < Nout; n0 += c.slice) {
    const int ns = Nout - n0 < c.slice ? Nout - n0 : c.slice;
    if (ns != c.gen.p.Cz) {
      if (const char* why = plan_generic(g, C0, C1, ns, Nout, out_f32, false, false, c.gen)) return fail(DCB_ERR_UNSUPPORTED, "%s", why);
    }
    TcFwdParams& p = c.gen.p;
    const void* Bs = reinterpret_cast<const __nv_bfloat16*>(B) + (size_t)n0 * wrow;
    void* o = reinterpret_cast<uint8_t*>(out) + (size_t)n0 * esz;
    p.relu = relu; p.out = reinterpret_cast<__nv_bfloat16*>(o);
    p.scale = scale ? scale + n0 : nullptr; p.shift = shift ? shift + n0 : nullptr;
    if (c.gen.pool) p.pool_out = reinterpret_cast<__nv_bfloat16*>(fuse->pool_out);
    if (c.gen.stats) p.stat_sums = stats->sums;
    const int swz = p.BK * 2;
    CUtensorMap mA0, mA1, mB;
    auto make_src_map = [&](CUtensorMap* m, const void* ptr, int C) -> int {
      if (p.mode == 0) return map_nhwc(m, g.f16, ptr, g.N, g.IH, g.IW, C, C, p.BK, p.bw, p.bh, p.bn, swz);
      if (p.mode == 1) return map_rows(m, g.f16, ptr, (long long)g.N * g.IH, g.IW, C, p.BK, p.bw, p.bh, swz);
      return map_subpixel(m, g.f16, ptr, (long long)g.N * g.GH, g.GW, C, C, p.BK, p.bw, p.bh, swz);   // dy [N][2h][2w][C]
    };
    if (int e = make_src_map(&mA0, s0, C0)) return e;
    if (C1 > 0) { if (int e = make_src_map(&mA1, s1, C1)) return e; }
    else mA1 = mA0;
    if (int e = map_weights(&mB, g.f16, Bs, g.ntaps * (C0 + C1), p.Ntot, p.BK, p.BN, swz)) return e;
    CUtensorMap mO = mB;
    if (p.tma_store) {
      const int e = p.mode == 0 ? map_nhwc(&mO, g.f16, o, g.N, g.OH, g.OW, ns, Nout, 32, p.bw, p.bh, p.bn, 64)
                                : map_subpixel(&mO, g.f16, o, (long long)g.N * g.GH, g.GW, ns, Nout, 32, p.bw, p.bh, 64);   // convT fwd y
      if (e) return e;
    }
    auto* k = c.gen.stats ? tapgemm_tc_fwd_kernel<false, true> : c.gen.pool ? tapgemm_tc_fwd_kernel<true, false>
                                                                           : tapgemm_tc_fwd_kernel<false, false>;
    if (int e = launch(k, "tapgemm_tc_fwd_kernel", c.gen.grid, TC_THREADS, c.gen.dyn, TC_SMEM_MAX, st, policy(DCB_POLICY_PDL) != 0,
                       0, mA0, mA1, mB, mO, p))
      return e;
  }
  return DCB_OK;
}

static int launch_flat(const TapGeom& g, FwdPlan& c, const void* s0, int C0, const void* s1, int C1, const void* B, int Nout,
                       void* out, const float* scale, const float* shift, int relu, cudaStream_t st, TcStats* stats) {
  TcFlatParams& p = c.flat.p;
  p.relu = relu; p.out = out; p.scale = scale; p.shift = shift;
  if (c.flat.stats) p.stat_sums = stats->sums;
  CUtensorMap mA0, mA1, mB;
  if (int e = map_nhwc(&mA0, g.f16, s0, g.N, g.IH, g.IW, C0, C0, 64, p.Wp, p.R, 1, 128)) return e;
  if (C1 > 0) { if (int e = map_nhwc(&mA1, g.f16, s1, g.N, g.IH, g.IW, C1, C1, 64, p.Wp, p.R, 1, 128)) return e; } else mA1 = mA0;
  if (int e = map_weights(&mB, g.f16, B, 9 * (C0 + C1), Nout, 64, p.wrows, 128)) return e;
  return launch(c.flat.stats ? tapgemm_tc_flat_kernel<true> : tapgemm_tc_flat_kernel<false>, "tapgemm_tc_flat_kernel", c.flat.grid,
                FL_THREADS, c.flat.dyn, FL_SMEM_MAX, st, policy(DCB_POLICY_PDL) != 0, 0, mA0, mA1, mB, p);
}

// fuse != nullptr: the caller wants the head and/or the 2x2 max-pool computed in the conv epilogue; returns
// DCB_ERR_UNSUPPORTED (without launching) when this layer shape cannot take the fused path.
int run_tc_fwd(const TapGeom& g, const void* s0, int C0, const void* s1, int C1, const void* B, int Nout, void* out,
               const float* scale, const float* shift, int relu, int out_f32, cudaStream_t st, const TcFusion* fuse, TcStats* stats) {
  if (stats) stats->done = 0;
  if (stats && (fuse || out_f32)) return fail(DCB_ERR_INVALID_ARGUMENT, "batch statistics: plain 16-bit forward only");
  if (C0 % 32 != 0 || C1 % 32 != 0 || Nout % 32 != 0)
    return fail(DCB_ERR_UNSUPPORTED, "bf16 tensor-core path needs channel counts that are multiples of 32 "
                "(got C0=%d C1=%d Cout=%d); use the fp32 check mode for other widths", C0, C1, Nout);
  FwdPlan c = choose_fwd(g, C0, C1, Nout, fuse, stats != nullptr, out_f32);
  int e = DCB_OK;
  switch (c.kind) {
    case FwdPlan::UNSUPPORTED: return fail(DCB_ERR_UNSUPPORTED, "%s", c.error);
    case FwdPlan::GENERIC: e = launch_generic(g, c, s0, C0, s1, C1, B, Nout, out, scale, shift, relu, out_f32, st, fuse, stats); break;
    case FwdPlan::FLAT: e = launch_flat(g, c, s0, C0, s1, C1, B, Nout, out, scale, shift, relu, st, stats); break;
    default: e = launch_strip(g, c, s0, C0, s1, C1, B, Nout, out, scale, shift, relu, out_f32, st, fuse, stats); break;
  }
  if (e) return e;
  if (stats) stats->done = c.stats ? 1 : 0;
  note_kernel(fwd_kernel_name(c));
  return DCB_OK;
}

// ====================================================================================== wgrad
// part[split][tap][k][n] = sum over the split's pixels of A(pixel, tap, k) * G(pixel, n)
// UMMA: D[128 k-channels x BN n-channels] += A_sm^T * G_sm with the PIXEL axis as the MMA K dimension.
// Both operands sit in shared memory exactly as TMA delivers an NHWC box ([pixel rows][CB channels],
// swizzled), i.e. MN-major for the MMA: column blocks of CB channels are LBO apart, 8-pixel groups SBO apart.
constexpr int WG_P = 64;            // pixels per pipeline stage (4 UMMA K-steps of 16)

struct TcWgradParams {
  int mode;                 // 0: conv3x3 (4-D halo box for A, 4-D box for G)  2: convT (5-D strided A, 3-D merged G)
  int N, GH, GW;
  int bw, bh, bn;           // pixel box (bw*bh*bn = WG_P); mode 2: bh rows of the merged axis
  int tiles_w, tiles_h, tiles_n;
  int ntaps;
  int dy[9], dx[9];
  int C0, C1, CB;           // gathered operand: channels per source, channels per TMA box
  int Nout, CBG, BN;        // per-position operand: channels, channels per TMA box, n tile
  int splits;
  int stages;
  float* part;              // [splits][ntaps][K][Nout]
};

__global__ void __launch_bounds__(WG_THREADS, 1)
tapgemm_tc_wgrad_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
                        const __grid_constant__ CUtensorMap mapG, const TcWgradParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ uint64_t bar_full[TC_MAX_STAGES], bar_empty[TC_MAX_STAGES], bar_tfull[2], bar_tempty[2];
  __shared__ uint32_t tmem_base_smem;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // 1024-byte alignment as an offset into the __shared__ array (an integer round trip would turn every later access
  // through this pointer into a generic-space load/store)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int K = p.C0 + p.C1;
  const int ktiles = (K + 127) / 128, ntiles = p.Nout / p.BN;
  const int num_ptiles = p.tiles_w * p.tiles_h * p.tiles_n;
  const int num_items = ktiles * ntiles * p.ntaps * p.splits;
  const uint32_t a_blk_bytes = WG_P * p.CB * 2, g_blk_bytes = WG_P * p.CBG * 2;
  const uint32_t a_bytes = WG_P * 128 * 2, g_bytes = WG_P * p.BN * 2;
  const uint32_t stage_bytes = a_bytes + g_bytes;
  const int a_blks = 128 / p.CB, g_blks = p.BN / p.CBG;
  uint32_t tmem_cols = 32;
  while (tmem_cols < 2u * p.BN) tmem_cols <<= 1;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapA0);
    if (p.C1 > 0) tma_prefetch_desc(&mapA1);
    tma_prefetch_desc(&mapG);
    for (int s = 0; s < p.stages; ++s) { mbar_init(&bar_full[s], 1); mbar_init(&bar_empty[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&bar_tfull[s], 1); mbar_init(&bar_tempty[s], 4); }
    mbar_fence_init();
  }
  if (warp == 1) { tmem_alloc(&tmem_base_smem, tmem_cols); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;

  // item -> (ktile, ntile, tap, split): ktile fastest so neighbouring CTAs share the G tile in L2
  auto decode = [&](int item, int& kt, int& nt, int& tap, int& split) {
    kt = item % ktiles; item /= ktiles;
    nt = item % ntiles; item /= ntiles;
    tap = item % p.ntaps; split = item / p.ntaps;
  };

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0; uint32_t phase = 0;
      for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
        int kt, nt, tap, split;
        decode(item, kt, nt, tap, split);
        const int pt0 = (int)(((long long)num_ptiles * split) / p.splits);
        const int pt1 = (int)(((long long)num_ptiles * (split + 1)) / p.splits);
        // real column blocks of this k tile
        int nreal = 0;
        for (int b = 0; b < a_blks; ++b) if (kt * 128 + b * p.CB < K) ++nreal;
        const uint32_t tx = nreal * a_blk_bytes + g_bytes;
        for (int pt = pt0; pt < pt1; ++pt) {
          const int tw = pt % p.tiles_w, th = (pt / p.tiles_w) % p.tiles_h, tn = pt / (p.tiles_w * p.tiles_h);
          const int w0 = tw * p.bw, h0 = th * p.bh, n0 = tn * p.bn;
          mbar_wait(&bar_empty[stage], phase ^ 1);
          uint8_t* sa = smem + (size_t)stage * stage_bytes;
          uint8_t* sg = sa + a_bytes;
          mbar_arrive_expect_tx(&bar_full[stage], tx);
          for (int b = 0; b < a_blks; ++b) {
            const int kg = kt * 128 + b * p.CB;
            if (kg >= K) break;
            const bool second = kg >= p.C0;
            const int c0 = second ? kg - p.C0 : kg;
            const CUtensorMap* mA = second ? &mapA1 : &mapA0;
            if (p.mode == 0) tma_load_4d(mA, &bar_full[stage], sa + b * a_blk_bytes, c0, w0 + p.dx[tap], h0 + p.dy[tap], n0);
            else tma_load_5d(mA, &bar_full[stage], sa + b * a_blk_bytes, c0, p.dx[tap], w0, p.dy[tap], h0);
          }
          for (int b = 0; b < g_blks; ++b) {
            const int c0 = nt * p.BN + b * p.CBG;
            if (p.mode == 0) tma_load_4d(&mapG, &bar_full[stage], sg + b * g_blk_bytes, c0, w0, h0, n0);
            else tma_load_3d(&mapG, &bar_full[stage], sg + b * g_blk_bytes, c0, w0, h0);
          }
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      const uint32_t idesc = make_idesc_bf16(128, p.BN, 1, 1);
      const uint32_t swz_a = (p.CB == 64) ? SWZ_128B : SWZ_64B, swz_g = (p.CBG == 64) ? SWZ_128B : SWZ_64B;
      const uint32_t sbo_a = 8u * p.CB * 2u, sbo_g = 8u * p.CBG * 2u;
      const uint64_t dbase_a = make_smem_desc(0, a_blk_bytes, sbo_a, swz_a), dbase_g = make_smem_desc(0, g_blk_bytes, sbo_g, swz_g);
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      // hoisted shared addresses + split-phase polling of the stage barriers (see tapgemm_tc_fwd_kernel): a stage is
      // only four MMAs, so the ~250-cycle barrier poll and the address arithmetic were most of this thread's time
      const uint32_t smem_a = smem_u32_pinned(smem), a_full = smem_u32_pinned(bar_full), a_empty = smem_u32_pinned(bar_empty);
      asm volatile(".reg .pred p_wfull;");
      bool pre = false;
      for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
        int kt, nt, tap, split;
        decode(item, kt, nt, tap, split);
        const int pt0 = (int)(((long long)num_ptiles * split) / p.splits);
        const int pt1 = (int)(((long long)num_ptiles * (split + 1)) / p.splits);
        mbar_wait(&bar_tempty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * p.BN);
        for (int pt = pt0; pt < pt1; ++pt) {
          {
            uint32_t ok = 0;
            if (pre) asm volatile("selp.u32 %0, 1, 0, p_wfull;" : "=r"(ok));
            if (!ok) mbar_wait_a(a_full + 8u * stage, phase);
            int ns = stage + 1; uint32_t np = phase;
            if (ns == p.stages) { ns = 0; np ^= 1u; }
            asm volatile("mbarrier.test_wait.parity.shared::cta.b64 p_wfull, [%0], %1;" ::"r"(a_full + 8u * ns), "r"(np) : "memory");
            pre = true;
          }
          tc_fence_after();
          const uint32_t sa = smem_a + (uint32_t)stage * (uint32_t)stage_bytes;
          const uint32_t sg = sa + a_bytes;
#pragma unroll
          for (int k = 0; k < WG_P / 16; ++k) {
            // 16 pixels = two 8-row groups further down the box
            const uint64_t da = dbase_a + ((sa + k * 2 * sbo_a) >> 4);
            const uint64_t dg = dbase_g + ((sg + k * 2 * sbo_g) >> 4);
            umma_bf16(d_tmem, da, dg, idesc, (pt > pt0 || k > 0) ? 1u : 0u);
          }
          umma_commit_a(a_empty + 8u * stage);
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&bar_tfull[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;             // k channel within the tile
    int acc = 0; uint32_t acc_phase = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
      int kt, nt, tap, split;
      decode(item, kt, nt, tap, split);
      const int pt0 = (int)(((long long)num_ptiles * split) / p.splits);
      const int pt1 = (int)(((long long)num_ptiles * (split + 1)) / p.splits);
      const int kg = kt * 128 + row;
      float* dst = p.part + (((size_t)split * p.ntaps + tap) * K + kg) * p.Nout + nt * p.BN;
      mbar_wait(&bar_tfull[acc], acc_phase);
      tc_fence_after();
      const uint32_t t_addr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * p.BN);
      for (int c = 0; c < p.BN; c += 32) {
        uint32_t r[32];
        tmem_ld_32x32b_x32(t_addr + c, r);
        tmem_ld_wait();
        if (kg < K) {
          // 32-byte stores: one full sector per lane and instruction (a lane owns an accumulator row, so a warp store
          // touches 32 different lines either way; as 16-byte stores the dump needed twice the requests)
          if (pt1 > pt0) {
#pragma unroll
            for (int j = 0; j < 32; j += 8)
              st_global_v8(dst + c + j, r[j], r[j + 1], r[j + 2], r[j + 3], r[j + 4], r[j + 5], r[j + 6], r[j + 7]);
          } else {                                   // empty split: nothing was accumulated
#pragma unroll
            for (int j = 0; j < 32; j += 8) st_global_v8(dst + c + j, 0, 0, 0, 0, 0, 0, 0, 0);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_tempty[acc]);
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) { tc_fence_after(); tmem_dealloc(tmem_base, tmem_cols); }
}

// ====================================================================================== wgrad strip kernel
// Weight gradient of the full-resolution 32-channel layers (enc0b, dec0a, dec0b: 3 of the 18 conv layers but
// two thirds of the generic wgrad time, because a 32-channel operand fills a quarter of the 128-row MMA and
// every tap re-loaded both operands).  Here:
//   * activation halo rows [66 px x 32 ch] stream through a ring exactly like the forward strip kernel;
//   * ONE MMA covers the three horizontal taps: the A operand is MN-major, its four 32-channel column blocks
//     are declared LBO = one pixel (64 B) apart, i.e. blocks 0..2 are the same halo row shifted by dx = 0..2
//     pixels (block 3 only feeds accumulator lanes 96..127, which are never read);
//   * the accumulators D[(dx, cin) x cout] for the 3 vertical taps (x sources) live in TMEM for the whole life
//     of the persistent CTA; each CTA writes a single partial at the end (fixed-order reduce afterwards).
constexpr int WS_PX = 64;             // pixels per step (4 MMA K-steps of 16)
constexpr int WS_RING = 8;            // halo rows in flight
constexpr int WS_GRING = 6;           // gradient rows in flight

struct TcWgradStripParams {
  int N, H, W;
  int nsrc;                 // 1 or 2 sources of 32 channels each
  int Nout;                 // 32 (64 B rows, SWIZZLE_64B) or 64 (128 B rows, SWIZZLE_128B)
  int R, wsegs, hchunks;
  int coff0, coff1;         // channel coordinate of each 32-channel block inside its tensor
  float* part;              // [gridDim.x][9][32 * nsrc][Nout]
};

__global__ void __launch_bounds__(WG_THREADS, 1)
tapgemm_tc_wgrad_strip_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
                              const __grid_constant__ CUtensorMap mapG, const TcWgradStripParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ uint64_t row_full[WS_RING], row_empty[WS_RING], g_full[WS_GRING], g_empty[WS_GRING], bar_done;
  __shared__ uint32_t tmem_base_smem;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // 1024-byte alignment as an offset into the __shared__ array (an integer round trip would turn every later access
  // through this pointer into a generic-space load/store)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  constexpr uint32_t A_SLOT = 5120;                       // 66 (+ spill) rows x 64 B, 1024-aligned
  const uint32_t row_bytes = (uint32_t)p.nsrc * A_SLOT;
  const uint32_t g_slot = (uint32_t)WS_PX * p.Nout * 2;   // 4 KB or 8 KB
  uint8_t* s_ring = smem;
  uint8_t* s_g = smem + (size_t)WS_RING * row_bytes;
  const int num_items = p.N * p.hchunks * p.wsegs;
  const int nacc = 3 * p.nsrc;
  uint32_t tmem_cols = 32;
  while (tmem_cols < (uint32_t)(nacc * p.Nout)) tmem_cols <<= 1;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapA0);
    if (p.nsrc > 1) tma_prefetch_desc(&mapA1);
    tma_prefetch_desc(&mapG);
    for (int i = 0; i < WS_RING; ++i) { mbar_init(&row_full[i], 1); mbar_init(&row_empty[i], 1); }
    for (int i = 0; i < WS_GRING; ++i) { mbar_init(&g_full[i], 1); mbar_init(&g_empty[i], 1); }
    mbar_init(&bar_done, 1);
    mbar_fence_init();
  }
  if (warp == 1) { tmem_alloc(&tmem_base_smem, tmem_cols); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;

  auto decode = [&](int item, int& n, int& h0, int& rows, int& w0) {
    const int ws = item % p.wsegs; item /= p.wsegs;
    const int hc = item % p.hchunks; n = item / p.hchunks;
    h0 = hc * p.R; rows = p.H - h0 < p.R ? p.H - h0 : p.R; w0 = ws * WS_PX;
  };

  if (warp == 0) {
    if (elect_one()) {
      int pos = 0, gpos = 0; uint32_t ep = 0xffffffffu, gp = 0xffffffffu;
      for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
        int n, h0, rows, w0;
        decode(item, n, h0, rows, w0);
        for (int rr = -1; rr <= rows; ++rr) {
          mbar_wait(&row_empty[pos], (ep >> pos) & 1u); ep ^= 1u << pos;
          mbar_arrive_expect_tx(&row_full[pos], (uint32_t)p.nsrc * 66u * 64u);
          for (int sidx = 0; sidx < p.nsrc; ++sidx)
            tma_load_4d(sidx ? &mapA1 : &mapA0, &row_full[pos], s_ring + (size_t)pos * row_bytes + sidx * A_SLOT,
                        sidx ? p.coff1 : p.coff0, w0 - 1, h0 + rr, n);
          if (++pos == WS_RING) pos = 0;
          if (rr >= 0 && rr < rows) {
            mbar_wait(&g_empty[gpos], (gp >> gpos) & 1u); gp ^= 1u << gpos;
            mbar_arrive_expect_tx(&g_full[gpos], g_slot);
            tma_load_4d(&mapG, &g_full[gpos], s_g + (size_t)gpos * g_slot, 0, w0, h0 + rr, n);
            if (++gpos == WS_GRING) gpos = 0;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      // A: MN-major, 64 B rows (SWIZZLE_64B); column blocks (32 channels) one pixel apart -> LBO = 64 B; 8-pixel groups SBO = 512 B
      const uint64_t dbase_a = make_smem_desc(0, 64, 512, SWZ_64B);
      const uint32_t g_pitch = (uint32_t)p.Nout * 2;
      const uint64_t dbase_g = make_smem_desc(0, g_slot, 8 * g_pitch, p.Nout == 64 ? SWZ_128B : SWZ_64B);
      const uint32_t idesc = make_idesc_bf16(128, p.Nout, 1, 1);
      const uint32_t ring16 = smem_u32(s_ring) >> 4, g16 = smem_u32(s_g) >> 4;
      const uint32_t rowb16 = row_bytes >> 4, gslot16 = g_slot >> 4;
      int pos_next = 0, gpos = 0; uint32_t fp = 0, gfp = 0;
      auto wait_next_row = [&]() -> int {
        const int ps = pos_next;
        mbar_wait(&row_full[ps], (fp >> ps) & 1u); fp ^= 1u << ps;
        pos_next = (ps + 1 == WS_RING) ? 0 : ps + 1;
        return ps;
      };
      uint32_t accf = 0;                                       // first MMA of every accumulator overwrites
      for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
        int n, h0, rows, w0;
        decode(item, n, h0, rows, w0);
        int p0 = wait_next_row(), p1 = wait_next_row();
        for (int t = 0; t < rows; ++t) {
          const int p2 = wait_next_row();
          mbar_wait(&g_full[gpos], (gfp >> gpos) & 1u); gfp ^= 1u << gpos;
          tc_fence_after();
          const uint32_t rows16[3] = {ring16 + p0 * rowb16, ring16 + p1 * rowb16, ring16 + p2 * rowb16};
          const uint64_t dg0 = dbase_g + (g16 + gpos * gslot16);
#pragma unroll
          for (int dy = 0; dy < 3; ++dy) {
            for (int sidx = 0; sidx < p.nsrc; ++sidx) {
              const uint32_t d_tmem = tmem_base + (uint32_t)((dy * p.nsrc + sidx) * p.Nout);
              const uint64_t da0 = dbase_a + (rows16[dy] + sidx * (A_SLOT >> 4));
#pragma unroll
              for (int k = 0; k < WS_PX / 16; ++k)            // 16 pixels further down: 16 rows of 64 B / of g_pitch
                umma_bf16(d_tmem, da0 + (uint64_t)(k * 64), dg0 + (uint64_t)(k * g_pitch), idesc, (accf | (uint32_t)k) ? 1u : 0u);
            }
          }
          accf = 1;
          umma_commit(&g_empty[gpos]);
          umma_commit(&row_empty[p0]);
          if (++gpos == WS_GRING) gpos = 0;
          p0 = p1; p1 = p2;
        }
        umma_commit(&row_empty[p0]);
        umma_commit(&row_empty[p1]);
      }
      umma_commit(&bar_done);
    }
  } else {
    // one dump of the accumulators at the very end: lane = dx * 32 + cin
    const int quarter = warp & 3;
    mbar_wait(&bar_done, 0);
    tc_fence_after();
    const bool has_work = blockIdx.x < num_items;
    const int K = 32 * p.nsrc;
    for (int a = 0; a < nacc; ++a) {
      const int dy = a / p.nsrc, sidx = a % p.nsrc;
      for (int c = 0; c < p.Nout; c += 32) {
        uint32_t r[32];
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(a * p.Nout + c), r);
        tmem_ld_wait();
        if (quarter < 3) {
          float* dst = p.part + (((size_t)blockIdx.x * 9 + (dy * 3 + quarter)) * K + sidx * 32 + lane) * p.Nout + c;
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            *reinterpret_cast<uint4*>(dst + j) = has_work ? make_uint4(r[j], r[j + 1], r[j + 2], r[j + 3]) : make_uint4(0, 0, 0, 0);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) { tc_fence_after(); tmem_dealloc(tmem_base, tmem_cols); }
}

void launch_reduce_splits(const float* part, int splits, size_t n, float* out, cudaStream_t st);
void launch_reduce_splits_rows(const float* part, int splits, int nrows, size_t row_len, float* out, size_t out_row_stride, cudaStream_t st);

struct WgradPlan { int BN, splits, CB, CBG, bw, bh, bn, tiles_w, tiles_h, tiles_n, stages; size_t ws_bytes; };

static WgradPlan plan_wgrad(const TapGeom& g, int K, int C0, int C1, int Nout) {
  WgradPlan w;
  const bool convT = (g.sy == 2);
  w.CB = (C0 % 64 == 0 && C1 % 64 == 0) ? 64 : 32;
  w.CBG = (Nout % 64 == 0) ? 64 : 32;
  w.BN = Nout < 256 ? Nout : 256;
  if (Nout % w.BN != 0) w.BN = 32;
  if (!convT) {
    w.bw = pick_pow2_box(g.GW, WG_P);
    w.bh = pick_pow2_box(g.GH, WG_P / w.bw);
    w.bn = WG_P / (w.bw * w.bh);
    w.tiles_w = cdiv(g.GW, w.bw); w.tiles_h = cdiv(g.GH, w.bh); w.tiles_n = cdiv(g.N, w.bn);
  } else {
    w.bw = pick_pow2_box(g.GW, WG_P);
    w.bh = WG_P / w.bw; w.bn = 1;
    w.tiles_w = cdiv(g.GW, w.bw); w.tiles_h = cdiv((long long)g.N * g.GH, w.bh); w.tiles_n = 1;
  }
  const int num_ptiles = w.tiles_w * w.tiles_h * w.tiles_n;
  const int base_items = cdiv(K, 128) * (Nout / w.BN) * g.ntaps;
  // two items per CTA, never a partial third wave: with the split count rounded UP, 9 x 33 = 297 items on 148 CTAs gave
  // one CTA three items and the launch the length of three (the static round-robin schedule has no stealing)
  int splits = (2 * sm_count()) / base_items;
  if (splits > num_ptiles) splits = num_ptiles;
  if (splits > 64) splits = 64;
  if (splits < 1) splits = 1;
  w.splits = splits;
  const size_t stage_bytes = (size_t)WG_P * 128 * 2 + (size_t)WG_P * w.BN * 2;
  int stages = (int)((200 * 1024) / stage_bytes);
  if (stages > TC_MAX_STAGES) stages = TC_MAX_STAGES;
  w.stages = stages;
  w.ws_bytes = (size_t)splits * g.ntaps * K * Nout * sizeof(float);
  return w;
}

// sources are consumed as 32-channel blocks (<= 2 per launch: 3 dy x 2 blocks x Nout accumulator columns <= 512);
// a 64-channel tensor is two blocks of the same tensor map, more than two blocks run as several launches
static bool wgrad_strip_ok(const TapGeom& g, int C0, int C1, int Nout) {
  return policy(DCB_POLICY_WGRAD_STRIP) && g.ntaps == 9 && g.sy == 1 && (C0 == 32 || C0 == 64) && (C1 == 0 || C1 == 32 || C1 == 64) &&
         (Nout == 32 || Nout == 64) && g.GW % WS_PX == 0;
}

size_t tc_wgrad_workspace(const TapGeom& g, int K, int Nout) {
  // C0/C1 split does not change the split count; use a conservative plan
  size_t ws = plan_wgrad(g, K, K, 0, Nout).ws_bytes;
  if (K % 32 == 0 && K <= 128 && wgrad_strip_ok(g, 32, 0, Nout)) {
    const size_t strip = (size_t)sm_count() * 9 * 64 * Nout * sizeof(float);   // one launch covers <= 64 channels
    if (strip > ws) ws = strip;
  }
  return ws;
}

struct WgradBlock { const void* ptr; int C; int coff; };   // a 32-channel block: tensor, its channel count, channel offset

// one launch over nblk (1 or 2) blocks; the result lands in rows [k_off, k_off + 32 * nblk) of dW[9][K_total][Nout]
static int run_tc_wgrad_strip(const TapGeom& g, const WgradBlock* blk, int nblk, const void* G, int Nout, float* dW, int k_off,
                              int K_total, void* ws, size_t ws_bytes, cudaStream_t st) {
  TcWgradStripParams p;
  memset(&p, 0, sizeof(p));
  p.N = g.N; p.H = g.GH; p.W = g.GW; p.nsrc = nblk; p.Nout = Nout;
  p.coff0 = blk[0].coff; p.coff1 = nblk > 1 ? blk[1].coff : 0;
  p.wsegs = g.GW / WS_PX;
  int R = 32;
  while (R > 8 && (long long)g.N * cdiv(g.GH, R) * p.wsegs < 3LL * sm_count()) R >>= 1;
  p.R = R; p.hchunks = cdiv(g.GH, R);
  const int items = p.N * p.hchunks * p.wsegs;
  const int grid = items < sm_count() ? items : sm_count();
  const int K = 32 * nblk;
  const size_t need = (size_t)grid * 9 * K * Nout * sizeof(float);
  if (!ws || ws_bytes < need) return fail(DCB_ERR_WORKSPACE, "wgrad (bf16 strip): workspace %zu B < required %zu B", ws_bytes, need);
  p.part = reinterpret_cast<float*>(ws);
  CUtensorMap mA0, mA1, mG;
  if (int e = map_nhwc(&mA0, g.f16, blk[0].ptr, g.N, g.IH, g.IW, blk[0].C, blk[0].C, 32, 66, 1, 1, 64)) return e;
  if (nblk > 1) { if (int e = map_nhwc(&mA1, g.f16, blk[1].ptr, g.N, g.IH, g.IW, blk[1].C, blk[1].C, 32, 66, 1, 1, 64)) return e; }
  else mA1 = mA0;
  if (int e = map_nhwc(&mG, g.f16, G, g.N, g.GH, g.GW, Nout, Nout, Nout, WS_PX, 1, 1, Nout * 2)) return e;
  const size_t dyn = (size_t)WS_RING * nblk * 5120 + (size_t)WS_GRING * WS_PX * Nout * 2 + 1024;
  if (int e = launch(tapgemm_tc_wgrad_strip_kernel, "tapgemm_tc_wgrad_strip_kernel", grid, WG_THREADS, dyn, 160 * 1024, st, false, 0,
                     mA0, mA1, mG, p))
    return e;
  launch_reduce_splits_rows(p.part, grid, 9, K * Nout, dW + (size_t)k_off * Nout, (size_t)K_total * Nout, st);
  g_launches += 1;
  DCB_LAUNCH_OK("reduce_splits_kernel");
  note_kernel("wgrad_strip");
  return DCB_OK;
}

int run_tc_wgrad(const TapGeom& g, const void* s0, int C0, const void* s1, int C1, const void* G, int Nout, float* dW,
                 void* ws, size_t ws_bytes, cudaStream_t st) {
  if (g.f16) return fail(DCB_ERR_UNSUPPORTED, "the fp16 mode is inference only: gradients are computed in bf16 (or fp32 check) mode");
  if (C0 % 32 != 0 || C1 % 32 != 0 || Nout % 32 != 0)
    return fail(DCB_ERR_UNSUPPORTED, "bf16 tensor-core wgrad needs channel counts that are multiples of 32 "
                "(got C0=%d C1=%d N=%d)", C0, C1, Nout);
  const int K = C0 + C1;
  if (wgrad_strip_ok(g, C0, C1, Nout)) {
    WgradBlock blocks[4]; int nb = 0;
    for (int c = 0; c < C0; c += 32) blocks[nb++] = WgradBlock{s0, C0, c};
    for (int c = 0; c < C1; c += 32) blocks[nb++] = WgradBlock{s1, C1, c};
    for (int b = 0; b < nb; b += 2) {
      const int n = nb - b < 2 ? nb - b : 2;
      if (int e = run_tc_wgrad_strip(g, blocks + b, n, G, Nout, dW, 32 * b, K, ws, ws_bytes, st)) return e;
    }
    return DCB_OK;
  }
  const WgradPlan w = plan_wgrad(g, K, C0, C1, Nout);
  if (!ws || ws_bytes < w.ws_bytes) return fail(DCB_ERR_WORKSPACE, "wgrad (bf16): workspace %zu B < required %zu B", ws_bytes, w.ws_bytes);
  const bool convT = (g.sy == 2);
  TcWgradParams p;
  memset(&p, 0, sizeof(p));
  p.mode = convT ? 2 : 0;
  p.N = g.N; p.GH = g.GH; p.GW = g.GW;
  p.bw = w.bw; p.bh = w.bh; p.bn = w.bn; p.tiles_w = w.tiles_w; p.tiles_h = w.tiles_h; p.tiles_n = w.tiles_n;
  p.ntaps = g.ntaps;
  for (int t = 0; t < g.ntaps; ++t) { p.dy[t] = g.dy[t]; p.dx[t] = g.dx[t]; }
  p.C0 = C0; p.C1 = C1; p.CB = w.CB; p.Nout = Nout; p.CBG = w.CBG; p.BN = w.BN;
  p.splits = w.splits; p.stages = w.stages; p.part = reinterpret_cast<float*>(ws);

  CUtensorMap mA0, mA1, mG;
  auto make_a = [&](CUtensorMap* m, const void* ptr, int C) -> int {
    if (!convT) return map_nhwc(m, g.f16, ptr, g.N, g.IH, g.IW, C, C, w.CB, w.bw, w.bh, w.bn, w.CB * 2);
    return map_subpixel(m, g.f16, ptr, (long long)g.N * g.GH, g.GW, C, C, w.CB, w.bw, w.bh, w.CB * 2);
  };
  if (int e = make_a(&mA0, s0, C0)) return e;
  if (C1 > 0) { if (int e = make_a(&mA1, s1, C1)) return e; } else mA1 = mA0;
  if (int e = convT ? map_rows(&mG, g.f16, G, (long long)g.N * g.GH, g.GW, Nout, w.CBG, w.bw, w.bh, w.CBG * 2)
                    : map_nhwc(&mG, g.f16, G, g.N, g.GH, g.GW, Nout, Nout, w.CBG, w.bw, w.bh, w.bn, w.CBG * 2))
    return e;
  const size_t stage_bytes = (size_t)WG_P * 128 * 2 + (size_t)WG_P * w.BN * 2;
  const size_t dyn_smem = w.stages * stage_bytes + 1024;
  const int num_items = cdiv(K, 128) * (Nout / w.BN) * g.ntaps * w.splits;
  const int grid = num_items < sm_count() ? num_items : sm_count();
  if (int e = launch(tapgemm_tc_wgrad_kernel, "tapgemm_tc_wgrad_kernel", grid, WG_THREADS, dyn_smem, TC_SMEM_MAX, st, false, 0,
                     mA0, mA1, mG, p))
    return e;
  launch_reduce_splits(p.part, w.splits, (size_t)g.ntaps * K * Nout, dW, st);
  g_launches += 1;
  DCB_LAUNCH_OK("reduce_splits_kernel");
  note_kernel("wgrad");
  return DCB_OK;
}

}  // namespace dcb
