// Neurofinder scoring on the device (datasets/nf.py:153-174 of the reference, restated in deepcalcium/datasets/nf.py):
// 8-connected region labelling numbered like scipy.ndimage.label(m != 0, structure=ones((3, 3))), per-region pixel
// counts and coordinate sums, the greedy centre matching of neurofinder.match(a, b, threshold=5) and the matched
// overlaps.  Plus the orientation + reflect pad of the fit validation windows (unet_2d_summary.py:62-120) and the truth
// mask summary of a dataset's per-neuron planes (unet_2d_summary.py:244-291), whose clusters the labelling finds.
//
// Images come in through a device table of 8 x int64 records {ptr, H, W, row stride, col stride, kind, 0, 0}: pixel
// (y, x) is element y * row_stride + x * col_stride of ptr (signed, in elements, so flips / rotations / crops are
// views).  kind 0: uint8, foreground = nonzero; 1: fp32 and 2: fp64, foreground = round(p) != 0, i.e. !(|p| <= 0.5)
// (NaN is foreground, as on the host).
//
// Labelling is union-find in which a union always links the larger root to the smaller linear index (atomicMin), so
// the root of a component is its first pixel in raster order: 32 x 32 tiles are labelled in shared memory, tile
// borders are merged in global memory, the forest is flattened, and an exclusive scan of the root flags over
// 1024-pixel chunks numbers the components in raster order of their first pixel - scipy's numbering.  Every count
// and coordinate sum is an integer, so nothing depends on the order of the atomics.
#include <algorithm>
#include <climits>

#include "elementwise.cuh"

namespace dcb {

namespace {

constexpr int kTile = 32;        // labelling tile: kTile x kTile pixels, one thread each
constexpr int kChunk = 1024;     // linear pixel chunk of the scan / statistics kernels, one thread each
constexpr int kCand = 4;         // nearest candidates kept per truth region
constexpr double kMatchThreshold = 5.0;

struct Meta {                    // per-image offsets, computed on the device by setup_kernel
  long long* pix_off;            // [n+1] first pixel of image i in the concatenated pixel arrays
  int* tile_off;                 // [n+1] first labelling tile
  int* chunk_off;                // [n+1] first scan chunk
};

__device__ __forceinline__ bool fg_at(const long long* __restrict__ d, int y, int x) {
  const long long off = (long long)y * d[3] + (long long)x * d[4];
  switch ((int)d[5]) {
    case 0: return reinterpret_cast<const uint8_t*>(d[0])[off] != 0;
    case 1: return !(fabsf(reinterpret_cast<const float*>(d[0])[off]) <= 0.5f);
    default: return !(fabs(reinterpret_cast<const double*>(d[0])[off]) <= 0.5);
  }
}

// largest i in [0, n) with off[i] <= c (off[0] == 0 <= c < off[n]); skips images without blocks
__device__ __forceinline__ int find_image(const int* __restrict__ off, int n, int c) {
  int lo = 0, hi = n;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (off[mid] <= c) lo = mid; else hi = mid;
  }
  return lo;
}

__device__ __forceinline__ int find_root(const int* L, int a) {
  const volatile int* V = L;
  int p = V[a];
  while (p != a) { a = p; p = V[a]; }
  return a;
}

// Playne & Hawick's lock-free union: the larger root is linked to the smaller one, retried until the link holds
__device__ __forceinline__ void unite(int* L, int a, int b) {
  bool done;
  do {
    a = find_root(L, a); b = find_root(L, b);
    if (a < b) { const int old = atomicMin(L + b, a); done = old == b; b = old; }
    else if (b < a) { const int old = atomicMin(L + a, b); done = old == a; a = old; }
    else done = true;
  } while (!done);
}

// exclusive scan of v over the block (blockDim.x a multiple of 32); *total receives the block sum
__device__ __forceinline__ int block_exclusive_scan(int v, int* warp_tot, int* total) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) warp_tot[w] = x;
  __syncthreads();
  if (w == 0) {
    int t = lane < nw ? warp_tot[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, t, o);
      if (lane >= o) t += y;
    }
    warp_tot[lane] = t;
  }
  __syncthreads();
  const int r = (w ? warp_tot[w - 1] : 0) + x - v;
  *total = warp_tot[nw - 1];
  __syncthreads();
  return r;
}

__global__ void setup_kernel(const long long* __restrict__ desc, int n, Meta m) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  long long p = 0; int t = 0, c = 0;
  for (int i = 0; i < n; ++i) {
    m.pix_off[i] = p; m.tile_off[i] = t; m.chunk_off[i] = c;
    const int H = (int)desc[8 * i + 1], W = (int)desc[8 * i + 2];
    p += (long long)H * W;
    t += ((H + kTile - 1) / kTile) * ((W + kTile - 1) / kTile);
    c += (int)(((long long)H * W + kChunk - 1) / kChunk);
  }
  m.pix_off[n] = p; m.tile_off[n] = t; m.chunk_off[n] = c;
}

// one 32 x 32 tile per block: union-find in shared memory over the backward neighbours inside the tile, then every
// foreground pixel stores its tile root as an image-linear index; background stores -1
__global__ void __launch_bounds__(kTile * kTile) local_label_kernel(const long long* __restrict__ desc, int n, Meta m,
                                                                  int* __restrict__ L) {
  __shared__ int s[kTile * kTile];
  const int img = find_image(m.tile_off, n, blockIdx.x);
  const long long* d = desc + 8 * img;
  const int H = (int)d[1], W = (int)d[2];
  const int tiles_x = (W + kTile - 1) / kTile, tt = blockIdx.x - m.tile_off[img];
  const int y0 = (tt / tiles_x) * kTile, x0 = (tt % tiles_x) * kTile;
  const int t = threadIdx.x, ly = t / kTile, lx = t % kTile, y = y0 + ly, x = x0 + lx;
  const bool in = y < H && x < W;
  const bool f = in && fg_at(d, y, x);
  s[t] = f ? t : -1;
  __syncthreads();
  if (f) {                                    // foreground entries stay >= 0 while other threads link them
    if (lx > 0 && s[t - 1] >= 0) unite(s, t, t - 1);
    if (ly > 0) {
      if (lx > 0 && s[t - kTile - 1] >= 0) unite(s, t, t - kTile - 1);
      if (s[t - kTile] >= 0) unite(s, t, t - kTile);
      if (lx < kTile - 1 && s[t - kTile + 1] >= 0) unite(s, t, t - kTile + 1);
    }
  }
  __syncthreads();
  if (in) {
    int v = -1;
    if (f) {
      const int r = find_root(s, t);
      v = (y0 + r / kTile) * W + x0 + r % kTile;
    }
    L[m.pix_off[img] + (long long)y * W + x] = v;
  }
}

// merge across tile borders: each foreground pixel unites with its backward neighbours that lie in another tile
__global__ void __launch_bounds__(kChunk) border_merge_kernel(const long long* __restrict__ desc, int n, Meta m,
                                                              int* __restrict__ L) {
  const int img = find_image(m.chunk_off, n, blockIdx.x);
  const int H = (int)desc[8 * img + 1], W = (int)desc[8 * img + 2];
  const long long p = (long long)(blockIdx.x - m.chunk_off[img]) * kChunk + threadIdx.x;
  if (p >= (long long)H * W) return;
  int* Li = L + m.pix_off[img];
  const int pi = (int)p, y = pi / W, x = pi % W;
  if (Li[pi] < 0) return;
  const bool ty = y > 0 && y % kTile == 0, tx = x > 0 && x % kTile == 0;
  if (tx && Li[pi - 1] >= 0) unite(Li, pi, pi - 1);
  if (y > 0) {
    if (x > 0 && (ty || tx) && Li[pi - W - 1] >= 0) unite(Li, pi, pi - W - 1);
    if (ty && Li[pi - W] >= 0) unite(Li, pi, pi - W);
    if (x + 1 < W && (ty || (x + 1) % kTile == 0) && Li[pi - W + 1] >= 0) unite(Li, pi, pi - W + 1);
  }
}

// every foreground pixel points straight at its root; cnt[chunk] = number of roots (component first pixels)
__global__ void __launch_bounds__(kChunk) flatten_count_kernel(const long long* __restrict__ desc, int n, Meta m,
                                                               int* __restrict__ L, int* __restrict__ cnt) {
  const int img = find_image(m.chunk_off, n, blockIdx.x);
  const long long HW = desc[8 * img + 1] * desc[8 * img + 2];
  const long long p = (long long)(blockIdx.x - m.chunk_off[img]) * kChunk + threadIdx.x;
  bool root = false;
  if (p < HW) {
    int* Li = L + m.pix_off[img];
    if (Li[p] >= 0) {
      const int r = find_root(Li, (int)p);
      Li[p] = r;
      root = r == (int)p;
    }
  }
  const int c = __syncthreads_count(root);
  if (threadIdx.x == 0) cnt[blockIdx.x] = c;
}

// exclusive scan of the chunk root counts in place (cnt[nchunks] = total); region_base[i] = global number of the first
// region of image i (region_base[n] = total)
__global__ void __launch_bounds__(1024) scan_kernel(int* __restrict__ cnt, int nchunks, Meta m, int n,
                                                    int* __restrict__ region_base) {
  __shared__ int warp_tot[32];
  int carry = 0;
  for (int base = 0; base < nchunks; base += blockDim.x) {
    const int i = base + threadIdx.x;
    const int v = i < nchunks ? cnt[i] : 0;
    int tot;
    const int e = block_exclusive_scan(v, warp_tot, &tot);
    if (i < nchunks) cnt[i] = carry + e;
    carry += tot;
  }
  if (threadIdx.x == 0) cnt[nchunks] = carry;
  __syncthreads();
  for (int i = threadIdx.x; i <= n; i += blockDim.x) region_base[i] = cnt[m.chunk_off[i]];
}

// R[root pixel] = global region number (raster order of first pixels within an image, images in table order)
__global__ void __launch_bounds__(kChunk) rank_kernel(const long long* __restrict__ desc, int n, Meta m,
                                                      const int* __restrict__ L, const int* __restrict__ cnt,
                                                      int* __restrict__ R) {
  __shared__ int warp_tot[32];
  const int img = find_image(m.chunk_off, n, blockIdx.x);
  const long long HW = desc[8 * img + 1] * desc[8 * img + 2];
  const long long p = (long long)(blockIdx.x - m.chunk_off[img]) * kChunk + threadIdx.x;
  const long long g = m.pix_off[img] + p;
  const bool root = p < HW && L[g] == (int)p;
  int tot;
  const int e = block_exclusive_scan(root ? 1 : 0, warp_tot, &tot);
  if (root) R[g] = cnt[blockIdx.x] + e;
}

// global region number of pixel p of image img, or -1 for background
__device__ __forceinline__ int region_of(const int* __restrict__ L, const int* __restrict__ R, long long pix_off, long long p) {
  const int l = L[pix_off + p];
  return l < 0 ? -1 : R[pix_off + l];
}

__global__ void __launch_bounds__(kChunk) write_labels_kernel(const long long* __restrict__ desc, int n, Meta m,
                                                              const int* __restrict__ L, const int* __restrict__ R,
                                                              const int* __restrict__ region_base, int* __restrict__ labels) {
  const int img = find_image(m.chunk_off, n, blockIdx.x);
  const long long HW = desc[8 * img + 1] * desc[8 * img + 2];
  const long long p = (long long)(blockIdx.x - m.chunk_off[img]) * kChunk + threadIdx.x;
  if (p >= HW) return;
  const int r = region_of(L, R, m.pix_off[img], p);
  labels[m.pix_off[img] + p] = r < 0 ? 0 : r - region_base[img] + 1;
}

// info[3 r] += pixel count, sr[r] += sum of rows, sc[r] += sum of columns; lanes of a warp on the same region add once
__global__ void __launch_bounds__(kChunk) stats_kernel(const long long* __restrict__ desc, int n, Meta m,
                                                       const int* __restrict__ L, const int* __restrict__ R,
                                                       int* __restrict__ info, unsigned long long* __restrict__ sr,
                                                       unsigned long long* __restrict__ sc) {
  const int img = find_image(m.chunk_off, n, blockIdx.x);
  const int W = (int)desc[8 * img + 2];
  const long long HW = desc[8 * img + 1] * W;
  const long long p = (long long)(blockIdx.x - m.chunk_off[img]) * kChunk + threadIdx.x;
  const int r = p < HW ? region_of(L, R, m.pix_off[img], p) : -1;
  const unsigned act = __ballot_sync(0xffffffffu, r >= 0);
  if (r < 0) return;
  const unsigned peers = __match_any_sync(act, r);
  const unsigned y = (unsigned)(p / W), x = (unsigned)(p % W);   // H, W < 2^24: 32 of them fit 32 bits
  const unsigned sy = __reduce_add_sync(peers, y), sx = __reduce_add_sync(peers, x);
  if ((int)(threadIdx.x & 31) == __ffs(peers) - 1) {
    atomicAdd(info + 3 * r, __popc(peers));
    atomicAdd(sr + r, (unsigned long long)sy);
    atomicAdd(sc + r, (unsigned long long)sx);
  }
}

// centre distance exactly as numpy evaluates sqrt(((targets - c) ** 2).sum(axis=1)): every step rounded on its own
__device__ __forceinline__ double centre_distance(double2 a, double2 b) {
  const double dy = __dsub_rn(b.x, a.x), dx = __dsub_rn(b.y, a.y);
  return __dsqrt_rn(__dadd_rn(__dmul_rn(dy, dy), __dmul_rn(dx, dx)));
}

// one block per pair: centres (exact integer sums divided once), then for every truth region the number of prediction
// regions closer than the threshold and the kCand nearest of them, ordered by (distance, region)
__global__ void __launch_bounds__(256) candidates_kernel(const int* __restrict__ region_base, int* __restrict__ info,
                                                         const unsigned long long* __restrict__ sr,
                                                         const unsigned long long* __restrict__ sc, double2* __restrict__ cen,
                                                         int* __restrict__ cand, int* __restrict__ ncand) {
  const int a0 = region_base[2 * blockIdx.x], a1 = region_base[2 * blockIdx.x + 1], b1 = region_base[2 * blockIdx.x + 2];
  for (int r = a0 + threadIdx.x; r < b1; r += blockDim.x) {
    const double c = (double)info[3 * r];
    cen[r] = make_double2((double)sr[r] / c, (double)sc[r] / c);
    info[3 * r + 1] = -1;
  }
  __syncthreads();
  for (int a = a0 + threadIdx.x; a < a1; a += blockDim.x) {
    const double2 ca = cen[a];
    double bd[kCand];
    int bb[kCand];
#pragma unroll
    for (int k = 0; k < kCand; ++k) { bd[k] = kMatchThreshold; bb[k] = -1; }
    int nc = 0;
    for (int b = a1; b < b1; ++b) {
      const double d = centre_distance(ca, cen[b]);
      if (!(d < kMatchThreshold)) continue;
      ++nc;
      if (d < bd[kCand - 1]) {              // b grows: among equal distances the earlier (smaller) region stays first
        bd[kCand - 1] = d; bb[kCand - 1] = b;
#pragma unroll
        for (int k = kCand - 1; k > 0; --k) {
          if (bd[k] < bd[k - 1]) {
            const double td = bd[k]; bd[k] = bd[k - 1]; bd[k - 1] = td;
            const int tb = bb[k]; bb[k] = bb[k - 1]; bb[k - 1] = tb;
          }
        }
      }
    }
#pragma unroll
    for (int k = 0; k < kCand; ++k) cand[(long long)a * kCand + k] = bb[k];
    ncand[a] = nc;
  }
}

// neurofinder.match, one thread per pair: truth regions in label order take the nearest remaining prediction region
// closer than the threshold (ties: the smaller label).  The first untaken entry of the sorted candidate list is that
// region; only when all kCand listed candidates are taken and more exist are the pair's prediction regions rescanned.
__global__ void greedy_match_kernel(const int* __restrict__ region_base, int n_pairs, const double2* __restrict__ cen,
                                    const int* __restrict__ cand, const int* __restrict__ ncand, uint8_t* __restrict__ taken,
                                    int* __restrict__ info) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pairs) return;
  const int a0 = region_base[2 * i], a1 = region_base[2 * i + 1], b1 = region_base[2 * i + 2];
  for (int a = a0; a < a1; ++a) {
    const int nc = ncand[a];
    int hit = -1;
    for (int k = 0; k < min(nc, kCand) && hit < 0; ++k) {
      const int b = cand[(long long)a * kCand + k];
      if (!taken[b]) hit = b;
    }
    if (hit < 0 && nc > kCand) {
      const double2 ca = cen[a];
      double best = kMatchThreshold;
      for (int b = a1; b < b1; ++b) {
        if (taken[b]) continue;
        const double d = centre_distance(ca, cen[b]);
        if (d < best) { best = d; hit = b; }
      }
    }
    if (hit >= 0) {
      taken[hit] = 1;
      info[3 * a + 1] = hit - a1;
    }
  }
}

// info[3 a + 2] = number of pixels of truth region a that lie in its matched prediction region
__global__ void __launch_bounds__(kChunk) overlap_kernel(const long long* __restrict__ desc, int n, Meta m,
                                                         const int* __restrict__ L, const int* __restrict__ R,
                                                         const int* __restrict__ region_base, int* __restrict__ info) {
  const int img = find_image(m.chunk_off, n, blockIdx.x);
  if (img & 1) return;
  const long long HW = desc[8 * img + 1] * desc[8 * img + 2];
  const long long p = (long long)(blockIdx.x - m.chunk_off[img]) * kChunk + threadIdx.x;
  if (p >= HW) return;
  const int a = region_of(L, R, m.pix_off[img], p);
  if (a < 0) return;
  const int hit = info[3 * a + 1];
  if (hit >= 0 && region_of(L, R, m.pix_off[img + 1], p) == region_base[img + 1] + hit) atomicAdd(info + 3 * a + 2, 1);
}

// ---- host side
struct Layout {
  long long npix = 0, rcap = 0;
  int ntiles = 0, nchunks = 0;
  size_t o_pix, o_tile, o_chunk, o_L, o_R, o_cnt, o_sr, o_sc, o_cen, o_cand, o_ncand, o_taken, bytes;
};

size_t align_up(size_t v) { return (v + 255) & ~(size_t)255; }

int make_layout(const long long* h_desc, int n, Layout& ly) {
  DCB_CHECK_ARG(h_desc && n > 0, "region labelling: no images");
  for (int i = 0; i < n; ++i) {
    const long long* d = h_desc + 8 * i;
    const long long H = d[1], W = d[2];
    DCB_CHECK_ARG(H >= 0 && W >= 0 && H < (1 << 24) && W < (1 << 24), "region labelling: image %d has shape %lld x %lld", i, H, W);
    DCB_CHECK_ARG(d[5] >= 0 && d[5] <= 2, "region labelling: image %d has kind %lld (0 uint8, 1 fp32, 2 fp64)", i, d[5]);
    DCB_CHECK_ARG(H * W == 0 || d[0] != 0, "region labelling: image %d has no data pointer", i);
    ly.npix += H * W;
    ly.rcap += ((H + 1) / 2) * ((W + 1) / 2);     // most 8-connected components an H x W image can hold
    ly.ntiles += (int)(((H + kTile - 1) / kTile) * ((W + kTile - 1) / kTile));
    ly.nchunks += (int)((H * W + kChunk - 1) / kChunk);
  }
  DCB_CHECK_ARG(ly.npix < (1ll << 31), "region labelling: %lld pixels in one call (at most 2^31 - 1)", ly.npix);
  size_t o = 0;
  auto take = [&](size_t bytes) { const size_t at = o; o = align_up(o + bytes); return at; };
  ly.o_pix = take(sizeof(long long) * (n + 1));
  ly.o_tile = take(sizeof(int) * (n + 1));
  ly.o_chunk = take(sizeof(int) * (n + 1));
  ly.o_L = take(sizeof(int) * ly.npix);
  ly.o_R = take(sizeof(int) * ly.npix);
  ly.o_cnt = take(sizeof(int) * (ly.nchunks + 1));
  ly.o_sr = take(sizeof(unsigned long long) * ly.rcap);
  ly.o_sc = take(sizeof(unsigned long long) * ly.rcap);
  ly.o_cen = take(sizeof(double2) * ly.rcap);
  ly.o_cand = take(sizeof(int) * kCand * ly.rcap);
  ly.o_ncand = take(sizeof(int) * ly.rcap);
  ly.o_taken = take(ly.rcap);
  ly.bytes = o;
  return DCB_OK;
}

template <typename T> T* at(void* ws, size_t off) { return reinterpret_cast<T*>(static_cast<char*>(ws) + off); }

// labels of every image -> L (roots), R (global region numbers of the roots), region_base
int label_core(const long long* desc, int n, const Layout& ly, void* ws, int* region_base, cudaStream_t st) {
  const Meta m{at<long long>(ws, ly.o_pix), at<int>(ws, ly.o_tile), at<int>(ws, ly.o_chunk)};
  int* L = at<int>(ws, ly.o_L); int* R = at<int>(ws, ly.o_R); int* cnt = at<int>(ws, ly.o_cnt);
  setup_kernel<<<1, 32, 0, st>>>(desc, n, m);
  DCB_LAUNCH_OK("setup_kernel");
  g_launches += 2;
  if (ly.npix > 0) {
    local_label_kernel<<<ly.ntiles, kTile * kTile, 0, st>>>(desc, n, m, L);
    DCB_LAUNCH_OK("local_label_kernel");
    border_merge_kernel<<<ly.nchunks, kChunk, 0, st>>>(desc, n, m, L);
    DCB_LAUNCH_OK("border_merge_kernel");
    flatten_count_kernel<<<ly.nchunks, kChunk, 0, st>>>(desc, n, m, L, cnt);
    DCB_LAUNCH_OK("flatten_count_kernel");
    g_launches += 3;
  }
  scan_kernel<<<1, 1024, 0, st>>>(cnt, ly.nchunks, m, n, region_base);
  DCB_LAUNCH_OK("scan_kernel");
  if (ly.npix > 0) {
    rank_kernel<<<ly.nchunks, kChunk, 0, st>>>(desc, n, m, L, cnt, R);
    DCB_LAUNCH_OK("rank_kernel");
    g_launches += 1;
  }
  return DCB_OK;
}

__global__ void orient_pad_kernel(const float* __restrict__ s, int hs, int ws, int k, int H, int W, float* __restrict__ out) {
  const int hf = (k == 3 || k == 5) ? ws : hs, wf = (k == 3 || k == 5) ? hs : ws;
  const long long total = (long long)H * W;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int a = reflect_index((int)(idx / W), hf), b = reflect_index((int)(idx % W), wf);
    int i, j;
    switch (k) {
      case 0: i = a; j = b; break;                       // identity
      case 1: i = a; j = ws - 1 - b; break;              // np.fliplr
      case 2: i = hs - 1 - a; j = b; break;              // np.flipud
      case 3: i = b; j = ws - 1 - a; break;              // np.rot90(s, 1)
      case 4: i = hs - 1 - a; j = ws - 1 - b; break;     // np.rot90(s, 2)
      default: i = hs - 1 - b; j = a; break;             // np.rot90(s, 3)
    }
    out[idx] = s[(long long)i * ws + j];
  }
}

// ---- mask summary (unet_2d_summary.py:244-291, _summarize_mask): masks [n][H][W] (one byte, "== 1" counts) -> [H][W]
// Only a candidate centre - an alive pixel whose alive 3 x 3 window holds two owners - ever deletes, and deletions only
// shrink windows.  Candidates in different 8-connected components of the 3 x 3 dilation of the candidate map are >= 4 px
// apart, so their windows are disjoint: each component (cluster) is walked on its own, in (owner, y, x) order.
constexpr int kZChunk = 64;      // planes per thread of the owner pass
constexpr int kSortCap = 2048;   // largest cluster sorted in shared memory

// packed[p] += {planes == 1 in this thread's chunk} << 32 | {that plane, when it is the only one}: the high word counts the
// planes (carries from the low word only ever raise a count that is already >= 2); count 1 leaves the owner in the low word.
// Thread = 16 consecutive pixels x kZChunk planes; block 0 also writes the labelling table record of the dilated map.
__global__ void __launch_bounds__(256) mask_owner_kernel(const uint8_t* __restrict__ masks, int n, long long HW, bool vec,
                                                         unsigned long long* __restrict__ packed, long long* __restrict__ desc,
                                                         const uint8_t* dil, int H, int W) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    desc[0] = (long long)dil; desc[1] = H; desc[2] = W; desc[3] = W; desc[4] = 1;
    desc[5] = desc[6] = desc[7] = 0;
  }
  const long long groups = (HW + 15) / 16;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= groups * ((n + kZChunk - 1) / kZChunk)) return;
  const long long g = t % groups, p0 = g * 16;
  const int z0 = (int)(t / groups) * kZChunk, z1 = min(n, z0 + kZChunk);
  uint32_t cnt[4] = {0, 0, 0, 0};                    // per-byte saturating counts of 16 pixels
  int own[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) own[j] = 0;
#pragma unroll 4
  for (int z = z0; z < z1; ++z) {
    const uint8_t* src = masks + (size_t)z * HW + p0;
    uint32_t w[4];
    if (vec) {
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(src));
      w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        w[k] = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b)
          if (p0 + 4 * k + b < HW) w[k] |= (uint32_t)src[4 * k + b] << (8 * b);
      }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t eq = __vcmpeq4(w[k], 0x01010101u);
      if (eq) {
        cnt[k] = __vaddus4(cnt[k], eq & 0x01010101u);
#pragma unroll
        for (int b = 0; b < 4; ++b)
          if ((eq >> (8 * b)) & 1u) own[4 * k + b] = z;
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const unsigned c = (cnt[j >> 2] >> (8 * (j & 3))) & 0xffu;
    if (c) atomicAdd(packed + p0 + j, ((unsigned long long)c << 32) | (c == 1 ? (unsigned)own[j] : 0u));
  }
}

__device__ __forceinline__ int owner_at(const unsigned long long* __restrict__ packed, int H, int W, int y, int x) {
  if (y < 0 || y >= H || x < 0 || x >= W) return -1;
  const unsigned long long v = packed[(long long)y * W + x];
  return (v >> 32) == 1 ? (int)(unsigned)v : -1;
}

// per pixel: own (owner or -1 when no plane or several planes claim it), out = alive, dil = 3 candidate, 1 within one
// pixel of a candidate, 0 otherwise.  A pixel's flag needs the owners of its 5 x 5 neighbourhood.
__global__ void __launch_bounds__(256) mask_candidates_kernel(const unsigned long long* __restrict__ packed, int H, int W,
                                                              int* __restrict__ own, uint8_t* __restrict__ out,
                                                              uint8_t* __restrict__ dil) {
  const long long HW = (long long)H * W;
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < HW; p += (long long)gridDim.x * blockDim.x) {
    const int y = (int)(p / W), x = (int)(p % W);
    int o[5][5];
#pragma unroll
    for (int i = 0; i < 5; ++i)
#pragma unroll
      for (int j = 0; j < 5; ++j) o[i][j] = owner_at(packed, H, W, y + i - 2, x + j - 2);
    bool near = false, self = false;
#pragma unroll
    for (int ci = 1; ci < 4; ++ci)
#pragma unroll
      for (int cj = 1; cj < 4; ++cj) {
        int mn = INT_MAX, mx = -1;
#pragma unroll
        for (int i = -1; i <= 1; ++i)
#pragma unroll
          for (int j = -1; j <= 1; ++j) {
            const int v = o[ci + i][cj + j];
            if (v >= 0) { mn = min(mn, v); mx = max(mx, v); }
          }
        const bool cand = o[ci][cj] >= 0 && mn < mx;
        near |= cand;
        if (ci == 2 && cj == 2) self = cand;
      }
    own[p] = o[2][2];
    out[p] = o[2][2] >= 0;
    dil[p] = self ? 3 : (near ? 1 : 0);
  }
}

// cluster of a candidate pixel = the region number of its dilated component
__global__ void __launch_bounds__(kChunk) mask_cluster_count_kernel(const uint8_t* __restrict__ dil, long long HW,
                                                                    const int* __restrict__ L, const int* __restrict__ R,
                                                                    int* __restrict__ ccount) {
  const long long p = (long long)blockIdx.x * kChunk + threadIdx.x;
  if (p < HW && dil[p] == 3) atomicAdd(ccount + R[L[p]], 1);
}

// coff[c] = first key of cluster c (exclusive scan over the clusters the labelling found); coff[nclus] = candidates
__global__ void __launch_bounds__(1024) mask_cluster_scan_kernel(const int* __restrict__ region_base,
                                                                 const int* __restrict__ ccount, int* __restrict__ coff) {
  __shared__ int warp_tot[32];
  const int nclus = region_base[1];
  int carry = 0;
  for (int base = 0; base < nclus; base += blockDim.x) {
    const int i = base + threadIdx.x;
    int tot;
    const int e = block_exclusive_scan(i < nclus ? ccount[i] : 0, warp_tot, &tot);
    if (i < nclus) coff[i] = carry + e;
    carry += tot;
  }
  if (threadIdx.x == 0) coff[nclus] = carry;
}

// keys of cluster c in coff[c]..coff[c+1] (unordered; the walk sorts them): owner << 32 | linear index
__global__ void __launch_bounds__(kChunk) mask_cluster_scatter_kernel(const uint8_t* __restrict__ dil, long long HW,
                                                                      const int* __restrict__ L, const int* __restrict__ R,
                                                                      const int* __restrict__ own, const int* __restrict__ coff,
                                                                      int* __restrict__ ccount,
                                                                      unsigned long long* __restrict__ keys) {
  const long long p = (long long)blockIdx.x * kChunk + threadIdx.x;
  if (p >= HW || dil[p] != 3) return;
  const int c = R[L[p]];
  const int slot = atomicSub(ccount + c, 1) - 1;
  keys[coff[c] + slot] = ((unsigned long long)(unsigned)own[p] << 32) | (unsigned long long)p;
}

// block-wide merge sort of n distinct keys: in each pass every key moves to (its index in its run) + (keys of the partner
// run that are smaller).  a and b are both shared or both global memory; returns the buffer that holds the result.
__device__ unsigned long long* block_sort_keys(unsigned long long* a, unsigned long long* b, int n) {
  for (int w = 1; w < n; w <<= 1) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const unsigned long long k = a[i];
      const int r = i / w, mine = r * w, other = (r ^ 1) * w, start = min(mine, other);
      int lo = other, hi = min(other + w, n);
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (a[mid] < k) lo = mid + 1; else hi = mid;
      }
      b[start + (i - mine) + (lo - other)] = k;
    }
    __syncthreads();
    unsigned long long* t = a; a = b; b = t;
  }
  return a;
}

// one block per cluster (grid-stride over the cluster count, read on the device): sort its keys - in shared memory when
// they fit, else in place in global memory against the scratch copy tmp - then one thread walks them in order and
// deletes every alive pixel of each window that still holds two owners
__global__ void __launch_bounds__(256) mask_walk_kernel(const int* __restrict__ region_base, const int* __restrict__ coff,
                                                        unsigned long long* keys, unsigned long long* tmp,
                                                        const int* __restrict__ own, int H, int W, uint8_t* alive) {
  __shared__ unsigned long long sa[kSortCap], sb[kSortCap];
  const int nclus = region_base[1];
  for (int c = blockIdx.x; c < nclus; c += gridDim.x) {
    const int k0 = coff[c], n = coff[c + 1] - k0;
    unsigned long long* sorted;
    if (n <= kSortCap) {
      for (int i = threadIdx.x; i < n; i += blockDim.x) sa[i] = keys[k0 + i];
      __syncthreads();
      sorted = block_sort_keys(sa, sb, n);
    } else {
      sorted = block_sort_keys(keys + k0, tmp + k0, n);
    }
    if (threadIdx.x == 0) {
      for (int i = 0; i < n; ++i) {
        const int p = (int)(unsigned)sorted[i], y = p / W, x = p % W;
        const int y0 = max(y - 1, 0), y1 = min(y + 1, H - 1), x0 = max(x - 1, 0), x1 = min(x + 1, W - 1);
        int mn = INT_MAX, mx = -1;
        for (int yy = y0; yy <= y1; ++yy)
          for (int xx = x0; xx <= x1; ++xx)
            if (alive[yy * W + xx]) { const int o = own[yy * W + xx]; mn = min(mn, o); mx = max(mx, o); }
        if (mn < mx)
          for (int yy = y0; yy <= y1; ++yy)
            for (int xx = x0; xx <= x1; ++xx) alive[yy * W + xx] = 0;
      }
    }
    __syncthreads();
  }
}

struct MaskLayout {
  Layout lab;
  long long HW = 0;
  size_t o_desc, o_base, o_packed, o_own, o_dil, o_ccount, o_coff, o_tmp, bytes;
};

int make_mask_layout(int n, int H, int W, MaskLayout& ml) {
  DCB_CHECK_ARG(n >= 0 && H >= 0 && W >= 0, "mask summary: bad shape %d x %d x %d", n, H, W);
  ml.HW = (long long)H * W;
  const long long h_desc[8] = {1, H, W, W, 1, 0, 0, 0};        // shapes only: the pointer is set on the device
  const int st = make_layout(h_desc, 1, ml.lab);
  if (st != DCB_OK) return st;
  size_t o = align_up(ml.lab.bytes);
  auto take = [&](size_t bytes) { const size_t at = o; o = align_up(o + bytes); return at; };
  ml.o_desc = take(8 * sizeof(long long));
  ml.o_base = take(2 * sizeof(int));
  ml.o_packed = take(sizeof(unsigned long long) * ml.HW);      // after the candidate pass: the cluster keys
  ml.o_own = take(sizeof(int) * ml.HW);
  ml.o_dil = take(ml.HW);
  ml.o_ccount = take(sizeof(int) * ml.lab.rcap);
  ml.o_coff = take(sizeof(int) * (ml.lab.rcap + 1));
  ml.o_tmp = take(sizeof(unsigned long long) * ml.HW);
  ml.bytes = o;
  return DCB_OK;
}

}  // namespace
}  // namespace dcb

using namespace dcb;

extern "C" int dcb_nf_score_workspace_bytes(const long long* h_desc, int n_images, size_t* bytes, long long* region_capacity) {
  DCB_CHECK_ARG(bytes && region_capacity, "dcb_nf_score_workspace_bytes: null output");
  Layout ly;
  const int st = make_layout(h_desc, n_images, ly);
  if (st != DCB_OK) return st;
  *bytes = ly.bytes;
  *region_capacity = ly.rcap;
  return DCB_OK;
}

extern "C" int dcb_label_regions(const long long* desc, const long long* h_desc, int n_images, int* labels, int* region_base,
                                 void* workspace, size_t workspace_bytes, dcb_stream_t stream) {
  DCB_CHECK_ARG(desc && labels && region_base, "dcb_label_regions: null pointer");
  Layout ly;
  int st = make_layout(h_desc, n_images, ly);
  if (st != DCB_OK) return st;
  if (!workspace || workspace_bytes < ly.bytes)
    return fail(DCB_ERR_WORKSPACE, "dcb_label_regions: workspace of %zu bytes, %zu needed", workspace_bytes, ly.bytes);
  const cudaStream_t s = (cudaStream_t)stream;
  st = label_core(desc, n_images, ly, workspace, region_base, s);
  if (st != DCB_OK || ly.npix == 0) return st;
  const Meta m{at<long long>(workspace, ly.o_pix), at<int>(workspace, ly.o_tile), at<int>(workspace, ly.o_chunk)};
  write_labels_kernel<<<ly.nchunks, kChunk, 0, s>>>(desc, n_images, m, at<int>(workspace, ly.o_L), at<int>(workspace, ly.o_R),
                                                     region_base, labels);
  g_launches += 1;
  DCB_LAUNCH_OK("write_labels_kernel");
  return DCB_OK;
}

extern "C" int dcb_nf_score(const long long* desc, const long long* h_desc, int n_pairs, int* region_base, int* region_info,
                            void* workspace, size_t workspace_bytes, dcb_stream_t stream) {
  DCB_CHECK_ARG(desc && region_base && region_info && n_pairs > 0, "dcb_nf_score: bad arguments");
  Layout ly;
  int st = make_layout(h_desc, 2 * n_pairs, ly);
  if (st != DCB_OK) return st;
  for (int i = 0; i < n_pairs; ++i)
    DCB_CHECK_ARG(h_desc[16 * i + 1] == h_desc[16 * i + 9] && h_desc[16 * i + 2] == h_desc[16 * i + 10],
                  "dcb_nf_score: pair %d has a %lld x %lld truth and a %lld x %lld prediction", i, h_desc[16 * i + 1],
                  h_desc[16 * i + 2], h_desc[16 * i + 9], h_desc[16 * i + 10]);
  if (!workspace || workspace_bytes < ly.bytes)
    return fail(DCB_ERR_WORKSPACE, "dcb_nf_score: workspace of %zu bytes, %zu needed", workspace_bytes, ly.bytes);
  const cudaStream_t s = (cudaStream_t)stream;
  const int n = 2 * n_pairs;
  void* ws = workspace;
  // accumulators: counts / matches / overlaps, coordinate sums, taken flags
  DCB_CUDA_OK(cudaMemsetAsync(region_info, 0, sizeof(int) * 3 * ly.rcap, s));
  DCB_CUDA_OK(cudaMemsetAsync(at<char>(ws, ly.o_sr), 0, ly.o_cen - ly.o_sr, s));
  DCB_CUDA_OK(cudaMemsetAsync(at<char>(ws, ly.o_taken), 0, ly.rcap, s));
  st = label_core(desc, n, ly, ws, region_base, s);
  if (st != DCB_OK) return st;
  const Meta m{at<long long>(ws, ly.o_pix), at<int>(ws, ly.o_tile), at<int>(ws, ly.o_chunk)};
  const int* L = at<int>(ws, ly.o_L); const int* R = at<int>(ws, ly.o_R);
  auto* sr = at<unsigned long long>(ws, ly.o_sr); auto* sc = at<unsigned long long>(ws, ly.o_sc);
  auto* cen = at<double2>(ws, ly.o_cen);
  int* cand = at<int>(ws, ly.o_cand); int* ncand = at<int>(ws, ly.o_ncand);
  if (ly.npix > 0) {
    stats_kernel<<<ly.nchunks, kChunk, 0, s>>>(desc, n, m, L, R, region_info, sr, sc);
    DCB_LAUNCH_OK("stats_kernel");
  }
  candidates_kernel<<<n_pairs, 256, 0, s>>>(region_base, region_info, sr, sc, cen, cand, ncand);
  DCB_LAUNCH_OK("candidates_kernel");
  greedy_match_kernel<<<cdiv(n_pairs, 64), 64, 0, s>>>(region_base, n_pairs, cen, cand, ncand, at<uint8_t>(ws, ly.o_taken),
                                                       region_info);
  DCB_LAUNCH_OK("greedy_match_kernel");
  g_launches += 3;
  if (ly.npix > 0) {
    overlap_kernel<<<ly.nchunks, kChunk, 0, s>>>(desc, n, m, L, R, region_base, region_info);
    DCB_LAUNCH_OK("overlap_kernel");
    g_launches += 2;
  }
  return DCB_OK;
}

extern "C" int dcb_mask_summary_workspace_bytes(int n, int H, int W, size_t* bytes) {
  DCB_CHECK_ARG(bytes, "dcb_mask_summary_workspace_bytes: null output");
  MaskLayout ml;
  const int st = make_mask_layout(n, H, W, ml);
  if (st != DCB_OK) return st;
  *bytes = n == 0 ? 0 : ml.bytes;
  return DCB_OK;
}

extern "C" int dcb_mask_summary(const uint8_t* masks, int n, int H, int W, uint8_t* out, void* workspace,
                                size_t workspace_bytes, dcb_stream_t stream) {
  MaskLayout ml;
  int st = make_mask_layout(n, H, W, ml);
  if (st != DCB_OK) return st;
  const cudaStream_t s = (cudaStream_t)stream;
  if (ml.HW == 0) return DCB_OK;
  DCB_CHECK_ARG(out && (n == 0 || masks), "dcb_mask_summary: null pointer");
  if (n == 0) {
    DCB_CUDA_OK(cudaMemsetAsync(out, 0, ml.HW, s));
    return DCB_OK;
  }
  if (!workspace || workspace_bytes < ml.bytes)
    return fail(DCB_ERR_WORKSPACE, "dcb_mask_summary: workspace of %zu bytes, %zu needed", workspace_bytes, ml.bytes);
  void* ws = workspace;
  long long* desc = at<long long>(ws, ml.o_desc);
  int* base = at<int>(ws, ml.o_base);
  auto* packed = at<unsigned long long>(ws, ml.o_packed);
  int* own = at<int>(ws, ml.o_own);
  uint8_t* dil = at<uint8_t>(ws, ml.o_dil);
  int* ccount = at<int>(ws, ml.o_ccount);
  int* coff = at<int>(ws, ml.o_coff);
  DCB_CUDA_OK(cudaMemsetAsync(packed, 0, sizeof(unsigned long long) * ml.HW, s));
  DCB_CUDA_OK(cudaMemsetAsync(ccount, 0, sizeof(int) * ml.lab.rcap, s));
  const bool vec = ml.HW % 16 == 0 && reinterpret_cast<uintptr_t>(masks) % 16 == 0;
  const long long threads = (ml.HW + 15) / 16 * cdiv(n, kZChunk);
  DCB_CHECK_ARG(threads / 256 < (1ll << 31), "dcb_mask_summary: %d x %d x %d masks are too many for one call", n, H, W);
  mask_owner_kernel<<<cdiv(threads, 256), 256, 0, s>>>(masks, n, ml.HW, vec, packed, desc, dil, H, W);
  DCB_LAUNCH_OK("mask_owner_kernel");
  const int cap = sm_count() * 8;
  mask_candidates_kernel<<<std::min(cdiv(ml.HW, 256), cap), 256, 0, s>>>(packed, H, W, own, out, dil);
  DCB_LAUNCH_OK("mask_candidates_kernel");
  g_launches += 2;
  st = label_core(desc, 1, ml.lab, ws, base, s);
  if (st != DCB_OK) return st;
  const int* L = at<int>(ws, ml.lab.o_L); const int* R = at<int>(ws, ml.lab.o_R);
  mask_cluster_count_kernel<<<ml.lab.nchunks, kChunk, 0, s>>>(dil, ml.HW, L, R, ccount);
  DCB_LAUNCH_OK("mask_cluster_count_kernel");
  mask_cluster_scan_kernel<<<1, 1024, 0, s>>>(base, ccount, coff);
  DCB_LAUNCH_OK("mask_cluster_scan_kernel");
  mask_cluster_scatter_kernel<<<ml.lab.nchunks, kChunk, 0, s>>>(dil, ml.HW, L, R, own, coff, ccount, packed);
  DCB_LAUNCH_OK("mask_cluster_scatter_kernel");
  mask_walk_kernel<<<(int)std::min<long long>(ml.lab.rcap, cap), 256, 0, s>>>(base, coff, packed,
                                                                      at<unsigned long long>(ws, ml.o_tmp), own, H, W, out);
  DCB_LAUNCH_OK("mask_walk_kernel");
  g_launches += 4;
  return DCB_OK;
}

extern "C" int dcb_orient_pad_f32(const float* s, int hs, int ws, int k, int H, int W, float* out, dcb_stream_t stream) {
  DCB_CHECK_ARG(s && out && hs > 0 && ws > 0 && k >= 0 && k < 6, "dcb_orient_pad_f32: bad arguments");
  const int hf = (k == 3 || k == 5) ? ws : hs, wf = (k == 3 || k == 5) ? hs : ws;
  DCB_CHECK_ARG(H >= hf && W >= wf, "dcb_orient_pad_f32: %d x %d output for a %d x %d oriented image", H, W, hf, wf);
  const long long total = (long long)H * W;
  const long long cap = (long long)sm_count() * 16, blocks = (total + 255) / 256;
  orient_pad_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, (cudaStream_t)stream>>>(s, hs, ws, k, H, W, out);
  g_launches += 1;
  DCB_LAUNCH_OK("orient_pad_kernel");
  return DCB_OK;
}
