/* dcb200 - C ABI of the B200-native deep-calcium UNet2DS hot path.
 *
 * Every entry point replaces one piece of arithmetic that the reference
 * (alexklibisz/deep-calcium) delegates to numpy/h5py or Keras-2.0.6/TF-1.2.1;
 * the reference file:line each one stands in for is cited on the declaration.
 * Conventions:
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless
 *     the parameter name starts with h_ ;
 *   - the caller owns every buffer (including workspaces); the library keeps no
 *     persistent device allocations; host-side it caches only shape-keyed TMA
 *     descriptors;
 *   - all work is enqueued on `stream` (a cudaStream_t), no host synchronisation,
 *     CUDA-graph capturable;
 *   - return 0 on success, a negative dcb_status otherwise; dcb_last_error()
 *     gives the thread-local message of the last failure.
 * Activations are NHWC; `dtype` selects fp32 ("check mode", CUDA-core kernels)
 * or bf16 (tcgen05/TMEM/TMA kernels, fp32 accumulate).
 */
#ifndef DCB200_H_
#define DCB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* dcb_stream_t; /* cudaStream_t */

enum dcb_status {
  DCB_OK = 0,
  DCB_ERR_INVALID_ARGUMENT = -1,
  DCB_ERR_CUDA = -2,
  DCB_ERR_WORKSPACE = -3,
  DCB_ERR_UNSUPPORTED = -4
};

/* DCB_F16: fp16 activations and weights on the same tcgen05 kind::f16 MMA (same rate as bf16, 10 mantissa bits): inference
 * only - the forward entry points, pooling, upsampling and the head accept it; the gradient entry points do not */
enum dcb_dtype { DCB_F32 = 0, DCB_BF16 = 1, DCB_F16 = 2 };

/* loss ids: unet_2d_summary.py:372-377 */
enum dcb_loss { DCB_LOSS_BCE = 0, DCB_LOSS_WBCE = 1, DCB_LOSS_DICE = 2, DCB_LOSS_DICESQ = 3 };

int dcb_version(void);
const char* dcb_last_error(void);
/* number of kernels this library has launched from the calling process (bench.py's gpu_launches) */
unsigned long long dcb_launch_count(void);

/* Dispatch policy of the contraction kernels.  Process-wide, read at every call (nothing is cached, no environment
 * variables): tests and sweeps pin a kernel variant with dcb_set_policy(), run, and dcb_reset_policy().  Defaults are the
 * measured choices (profiles/).  dcb_last_kernel() names the variant the calling thread's last contraction call used,
 * e.g. "strip_fold", "strip", "strip_swap", "flat", "generic", "generic_swap", "wgrad", "wgrad_strip". */
enum dcb_policy_key {
  DCB_POLICY_FLAT = 0,          /* flat halo-tile conv kernel: 0 never, 1 auto (size gate), 2 whenever the shape is eligible */
  DCB_POLICY_STRIP = 1,         /* halo-strip conv kernel: 0 off, 1 on */
  DCB_POLICY_FOLD = 2,          /* vertical-tap folding inside the strip kernel: 0 off, 1 on */
  DCB_POLICY_NSPLIT = 3,        /* channel-split strip conv when the weights do not fit: 0 off, 1 one launch of two-CTA clusters sharing the halo rows by TMA multicast, 2 two launches */
  DCB_POLICY_SWAP_MIN_COUT = 4, /* smallest Cout that uses the weights-as-A orientation (0 = never) */
  DCB_POLICY_WGRAD_STRIP = 5,   /* strip weight-gradient kernel: 0 off, 1 on */
  DCB_POLICY_BN_CTAS_PER_SM = 6,
  DCB_POLICY_PROJ_I16_SPLITS = 7, /* T splits of the int16 projection (0 = heuristic) */
  DCB_POLICY_SPLITK = 8,        /* split-K of the generic conv kernel for small pixel counts: 0 off, 1 auto */
  DCB_POLICY_FUSED_BN = 9,      /* training BatchNorm: 0 = separate passes, 1 = single-launch kernels with grid barriers, 2 = batch statistics
                                   taken in the producing conv's epilogue where that is measured to pay (dcb_conv*_fwd_stats), 3 = wherever
                                   a statistics epilogue exists */
  DCB_POLICY_TMA_STORE = 10,    /* epilogues stage 16-bit outputs in shared memory and store them with TMA: 0 off, 1 convT forward, 2 also conv3x3 on the generic kernel */
  DCB_POLICY_BN_SLAB = 11,      /* training BatchNorm as channel-slab cluster kernels (DSMEM reduction): 0 off, 1 small tensors (measured gate), 2 wherever eligible */
  DCB_POLICY_PDL = 12,          /* programmatic dependent launch of the forward conv / TTA kernels: 0 off, 1 on.  Turn on only while
                                   enqueueing work whose per-channel scale / shift / weights are NOT written by kernels of the same
                                   stream sequence (inference): prologues read them before the dependency wait */
  DCB_POLICY_PAIR = 13,         /* folded strip conv on CTA-pair MMAs (tcgen05 cta_group::2, clusters of two): 0 off, 1 on */
  DCB_POLICY_COUNT = 14
};
int dcb_set_policy(int key, int value);
int dcb_get_policy(int key, int* value);
int dcb_reset_policy(void);
const char* dcb_last_kernel(void);

/* ---- a1: datasets/nf.py:115-130 (twin: examples/neurons/unet2ds_sj.py:67-85) ----
 * Per-pixel temporal mean and max of movie[T][H][W] (float32).  mean/max are
 * float32 [H][W].  floor_max_at_zero != 0 reproduces the reference's
 * zero-initialised running max (nf.py:125,130).  Sums are float64 internally. */
int dcb_proj_workspace_bytes(int T, int H, int W, size_t* bytes);
int dcb_proj_mean_max_f32(const float* movie, int T, int H, int W, float* mean, float* max,
                          int floor_max_at_zero, void* workspace, size_t workspace_bytes,
                          dcb_stream_t stream);
/* tuning hook used by bench/sweeps: variant<0 = default heuristic */
int dcb_proj_mean_max_f32_variant(const float* movie, int T, int H, int W, float* mean, float* max,
                                  int floor_max_at_zero, void* workspace, size_t workspace_bytes,
                                  int variant, int t_splits, dcb_stream_t stream);

/* same projection for an int16 movie (the reference's TIFF frames, datasets/nf.py:115-130): exact integer sums, half the bytes;
 * workspace as for the fp32 entry (dcb_proj_workspace_bytes) */
int dcb_proj_mean_max_i16(const short* movie, int T, int H, int W, float* mean, float* mx, int floor_max_at_zero, void* workspace,
                          size_t workspace_bytes, dcb_stream_t stream);
/* Streaming form for ingest (frames arrive in chunks, datasets/nf.py:126-130): accumulate a chunk of Tc int16 frames into
 * the per-pixel running state on the device - sum (int64, caller zero-initialises) and mx (int32, caller initialises to
 * INT_MIN) - then turn the state after T frames into the float32 mean / max images */
int dcb_proj_accum_i16(const short* chunk, int Tc, int H, int W, long long* sum, int* mx, dcb_stream_t stream);
int dcb_proj_accum_finalize(const long long* sum, const int* mx, int T, int H, int W, float* mean, float* max_out,
                            int floor_max_at_zero, dcb_stream_t stream);
/* same, for frames that were shifted by -bias before accumulation (unsigned 16-bit TIFF pixels, bias = 32768: the reference
 * computes mean / max from the unwrapped values, datasets/nf.py:129-130); the bias is restored in exact integer arithmetic */
int dcb_proj_accum_finalize_biased(const long long* sum, const int* mx, int T, int H, int W, int bias, float* mean,
                                   float* max_out, int floor_max_at_zero, dcb_stream_t stream);
/* ---- a2: unet_2d_summary.py:238-239 (_summarize_series) ----
 * out = (in - mean(in)) / std(in), population std, n = H*W elements.
 * stats (optional, 2 doubles on device) receives mean and std. */
int dcb_standardize_f32(const float* in, long long n, float* out, double* stats, dcb_stream_t stream);

/* ---- a3/a4/a8: every Conv2D(3x3,'same') / Conv2DTranspose(2x2,s2) of unet() and their
 * Keras-autodiff gradients (unet_2d_summary.py:154-167; arithmetic in TF 1.2.1).
 * Activations NHWC.  The input may be the channel concatenation [src0 | src1]
 * (unet_2d_summary.py:200,206,212,218); pass src1 = NULL, C1 = 0 otherwise.
 * Epilogue: out = act(acc * scale[c] + shift[c]) with scale/shift optional (NULL = 1 / 0)
 * and relu != 0 selecting max(0, .): inference folds bias + BatchNorm (eps 1e-3) + ReLU
 * into it, training passes shift = bias only and normalises after the batch statistics.
 *
 * Weight layouts (prepared once per weight update by dcb_prep_* below):
 *   DCB_F32 : conv3x3  B[9][Cin][Cout]   (= Keras HWIO)     convT fwd  B[4][Cin][Cout]
 *             conv3x3 dgrad B[9][Cout][Cin] (taps flipped)  convT dgrad B[4][Cout][Cin] (= Keras)
 *   DCB_BF16: the same matrices stored N-major ("K-major B"): [taps][N][K] -> see dcb_prep_*.
 */
int dcb_conv3x3_fwd(int dtype, const void* src0, int C0, const void* src1, int C1, int N, int H, int W,
                    const void* wgt, int Cout, const float* scale, const float* shift, int relu,
                    void* out, dcb_stream_t stream);
/* conv3x3 + epilogue with the next memory-bound op(s) of the graph folded in, so their input is not re-read
 * (and, for the head, never written): the 2x2/2 max-pool that follows an encoder block
 * (unet_2d_summary.py:176,182,188,194) and/or the 1x1 softmax head (:221-222).  `out` must always be a valid
 * [N][H][W][Cout] buffer; with need_y = 0 the library may leave it untouched.  Shapes the fused tensor-core
 * epilogue does not cover (and the fp32 check mode) run the unfused composition with identical results. */
typedef struct dcb_conv_fusion {
  const float* head_kernel; /* [Cout][2] or NULL */
  const float* head_bias;   /* [2] */
  float* logit;             /* [N*H*W] z1 - z0, may be NULL */
  float* prob;              /* [N*H*W] softmax(z)[1], may be NULL */
  int need_y;               /* 0: the caller never reads `out` */
  void* pool_out;           /* [N][H/2][W/2][Cout] or NULL */
} dcb_conv_fusion_t;
int dcb_conv3x3_fwd_fused(int dtype, const void* src0, int C0, const void* src1, int C1, int N, int H, int W,
                          const void* wgt, int Cout, const float* scale, const float* shift, int relu,
                          void* out, const dcb_conv_fusion_t* fuse, dcb_stream_t stream);
/* input h x w -> output 2h x 2w */
int dcb_convT2x2_fwd(int dtype, const void* src, int Cin, int N, int h, int w, const void* wgt, int Cout,
                     const float* scale, const float* shift, int relu, void* out, dcb_stream_t stream);
/* Training forward with the BatchNorm batch statistics taken in the conv epilogue (Keras BatchNormalization in training
 * mode normalises with the batch mean / biased variance, unet_2d_summary.py:157,165).  sums_q[0..Cout) += sum over all
 * output pixels of the STORED (rounded) output, sums_q[Cout..2 Cout) += sum of its squares, as 64-bit FIXED POINT in units
 * of 2^-20: per-CTA fp32 sums (fixed order) are added with integer atomics, so the totals are bit-reproducible whatever
 * the arrival order (range |total| < 8.8e12).  The caller ZEROES sums_q before the call.
 * *stats_done = 1 when the dispatched kernel accumulated into sums_q; 0 when this shape / dtype has no statistics
 * epilogue - the convolution has run all the same and the caller takes the statistics with its own pass
 * (dcb_bn_train_fwd).  Feeds dcb_bn_train_fwd_sums. */
int dcb_conv3x3_fwd_stats(int dtype, const void* src0, int C0, const void* src1, int C1, int N, int H, int W,
                          const void* wgt, int Cout, const float* scale, const float* shift, int relu, void* out,
                          long long* sums_q, int* stats_done, dcb_stream_t stream);
int dcb_convT2x2_fwd_stats(int dtype, const void* src, int Cin, int N, int h, int w, const void* wgt, int Cout,
                           const float* scale, const float* shift, int relu, void* out, long long* sums_q,
                           int* stats_done, dcb_stream_t stream);
int dcb_conv3x3_c1_fwd_stats(int dtype, const float* x, int N, int H, int W, const float* w, int Cout,
                             const float* scale, const float* shift, int relu, void* out, long long* sums_q,
                             int* stats_done, dcb_stream_t stream);
/* input gradients.  dy is the gradient w.r.t. the raw conv output in the activation dtype (it feeds the
 * tensor cores); dx is ALWAYS fp32: gradient tensors stay fp32 between layers because the BatchNorm
 * backward subtracts their per-channel mean (a bf16-rounded dx would lose most of its significant bits
 * there).  wgt is the *_dgrad operand of dcb_prep_*. */
int dcb_conv3x3_dgrad(int dtype, const void* dy, int Cout, int N, int H, int W, const void* wgt_dgrad, int Cin,
                      float* dx, dcb_stream_t stream);
/* dy is [N][2h][2w][Cout]; dx is [N][h][w][Cin] */
int dcb_convT2x2_dgrad(int dtype, const void* dy, int Cout, int N, int h, int w, const void* wgt, int Cin,
                       float* dx, dcb_stream_t stream);
/* dW[9][Cin][Cout] (fp32, Keras HWIO) = sum over pixels of x (shifted) * dy ; x may be [src0|src1] */
int dcb_conv3x3_wgrad_workspace_bytes(int dtype, int N, int H, int W, int Cin, int Cout, size_t* bytes);
int dcb_conv3x3_wgrad(int dtype, const void* src0, int C0, const void* src1, int C1, int N, int H, int W,
                      const void* dy, int Cout, float* dW, void* workspace, size_t workspace_bytes,
                      dcb_stream_t stream);
/* dW[2][2][Cout][Cin] (fp32, Keras layout); x is [N][h][w][Cin], dy is [N][2h][2w][Cout] */
int dcb_convT2x2_wgrad_workspace_bytes(int dtype, int N, int h, int w, int Cin, int Cout, size_t* bytes);
int dcb_convT2x2_wgrad(int dtype, const void* x, int Cin, int N, int h, int w, const void* dy, int Cout,
                       float* dW, void* workspace, size_t workspace_bytes, dcb_stream_t stream);
/* first layer (unet_2d_summary.py:169-172): 1-channel fp32 image x[N][H][W], w[9][Cout] fp32 (Keras
 * HWIO with Cin = 1), CUDA-core kernel (K = 9 is below any tensor-core tile); same epilogue as above */
int dcb_conv3x3_c1_fwd(int dtype, const float* x, int N, int H, int W, const float* w, int Cout,
                       const float* scale, const float* shift, int relu, void* out, dcb_stream_t stream);
int dcb_conv3x3_c1_wgrad_workspace_bytes(int Cout, size_t* bytes);
int dcb_conv3x3_c1_wgrad(int dtype, const float* x, const void* dy, int N, int H, int W, int Cout, float* dW,
                         void* workspace, size_t workspace_bytes, dcb_stream_t stream);
/* weight preparation from the fp32 Keras-layout master copies.
 *   conv3x3: w [3][3][Cin][Cout] -> fwd and dgrad operands for `dtype` (either may be NULL)
 *   convT  : w [2][2][Cout][Cin] -> fwd and dgrad operands */
int dcb_prep_conv3x3_weights(int dtype, const float* w, int Cin, int Cout, void* w_fwd, void* w_dgrad,
                             dcb_stream_t stream);
int dcb_prep_convT2x2_weights(int dtype, const float* w, int Cin, int Cout, void* w_fwd, void* w_dgrad,
                              dcb_stream_t stream);
/* every layer of a model in one launch.  desc_dev: device array of `count` records of 5 x int64
 * {w (fp32 master), w_fwd or 0, w_dgrad or 0, Cin | Cout << 32, kind: 0 = conv3x3 (HWIO), 1 = convT2x2 (2,2,Cout,Cin)};
 * layouts written exactly as by the two single-layer calls above */
int dcb_prep_weights_batch(int dtype, const long long* desc_dev, int count, dcb_stream_t stream);

/* ---- BatchNormalization (Keras 2.0.6: eps 1e-3, biased batch variance) ---- */
/* inference fold: scale = gamma*rsqrt(var+eps), shift = beta + (bias - mean)*scale */
int dcb_bn_fold(const float* gamma, const float* beta, const float* mean, const float* var, const float* bias,
                int C, float eps, float* scale, float* shift, dcb_stream_t stream);
/* sums[0..C) += sum_m x, sums[C..2C) += sum_m x^2 over x[M][C] (double; caller zeroes) */
int dcb_bn_stats(int dtype, const void* x, long long M, int C, double* sums, dcb_stream_t stream);
/* batch mean / rstd, scale/shift for dcb_bn_apply, momentum update of the moving statistics
 * (moving_* may be NULL) */
int dcb_bn_finalize(const double* sums, long long M, int C, const float* gamma, const float* beta, float eps,
                    float momentum, float* moving_mean, float* moving_var, float* scale, float* shift,
                    float* mean, float* rstd, dcb_stream_t stream);
/* y = relu?(x*scale + shift), then inverted dropout (Philox keyed by seed ^ *seed_dev and layer; p_drop = 0 disables;
 * unet_2d_summary.py:179-216) */
int dcb_bn_apply(int dtype, const void* x, long long M, int C, const float* scale, const float* shift, int relu,
                 float p_drop, unsigned long long seed, const unsigned long long* seed_dev, unsigned layer, void* y,
                 dcb_stream_t stream);
/* dcb_bn_finalize + dcb_bn_apply in one launch (training forward): the statistics of M_total rows (0 = M; the
 * data-parallel caller all-reduces `sums` first) become scale / shift inside the kernel */
int dcb_bn_finalize_apply(int dtype, const void* x, long long M, int C, const double* sums, long long M_total,
                          const float* gamma, const float* beta, float eps, float momentum, float* moving_mean,
                          float* moving_var, float* scale, float* shift, float* mean, float* rstd, int relu,
                          float p_drop, unsigned long long seed, const unsigned long long* seed_dev, unsigned layer,
                          void* y, dcb_stream_t stream);
/* backward of dropout+ReLU+BN given dy (fp32, row stride ldy, channel offset offy) and the raw conv output x:
 * reduce accumulates sums[0..C)=sum dz, sums[C..2C)=sum dz*xhat; apply writes d_raw and dgamma/dbeta.
 * Data-parallel use: all-reduce `sums` between the two calls, pass M_total = rows over all ranks
 * (0 = M) and dgb_scale = 1/world so that the later gradient all-reduce(sum) restores dgamma/dbeta */
int dcb_bn_bwd_reduce(int dtype, const float* dy, int ldy, int offy, const void* x, long long M, int C,
                      const float* scale, const float* shift, const float* mean, const float* rstd,
                      float p_drop, unsigned long long seed, const unsigned long long* seed_dev, unsigned layer,
                      double* sums, dcb_stream_t stream);
int dcb_bn_bwd_apply(int dtype, const float* dy, int ldy, int offy, const void* x, long long M, int C,
                     const float* scale, const float* shift, const float* mean, const float* rstd,
                     float p_drop, unsigned long long seed, const unsigned long long* seed_dev, unsigned layer,
                     const double* sums, long long M_total, float dgb_scale, void* draw, float* dgamma,
                     float* dbeta, dcb_stream_t stream);

/* ---- training BatchNorm as single-launch kernels (csrc/bn_fused.cu) ----
 * dcb_bn_train_fwd = dcb_bn_stats + dcb_bn_finalize_apply (+ dcb_maxpool2x2 when pool_out is given: N x H x W pixels,
 * M = N*H*W) in one persistent launch with one grid barrier; dcb_bn_train_bwd = dcb_bn_bwd_reduce + dcb_bn_bwd_apply
 * (draw may alias x).  Cross-CTA totals are 64-bit fixed-point integer sums (bit-reproducible, no floating-point atomics;
 * forward 2^-20 units, backward 2^-40 units).
 * workspace: dcb_bn_train_workspace_bytes(C) bytes that the caller ZEROES ONCE before the first use - the kernels leave it
 * zeroed, one workspace serves any number of stream-ordered launches; sync: 4 uint32 words that the caller zeroes before
 * EVERY launch.
 * peers (optional, data-parallel SyncBN): every rank's per-channel totals are exchanged inside the kernel through
 * peer-mapped memory (NVLink) and summed in rank order; M_total = rows over all ranks. */
typedef struct dcb_peer_exchange {
  int world, rank;                      /* <= 8 ranks */
  void* xchg[8];                        /* rank p's exchange area as mapped into THIS process (doubles) */
  void* flags[8];                       /* rank p's flag area as mapped into this process (uint64, zero-initialised) */
  long long slot_doubles;               /* doubles per slot, >= world * 2 * C */
  int slot;                             /* slot of this call: distinct per (layer, direction) within a step */
  const unsigned long long* epoch_dev;  /* device word that changes every step (state[0] of dcb_step_advance) */
} dcb_peer_exchange_t;
int dcb_bn_train_workspace_bytes(int C, size_t* bytes);
int dcb_bn_train_fwd(int dtype, const void* x, long long M, int C, long long M_total, const float* gamma,
                     const float* beta, float eps, float momentum, float* moving_mean, float* moving_var,
                     float* scale, float* shift, float* mean, float* rstd, int relu, float p_drop,
                     unsigned long long seed, const unsigned long long* seed_dev, unsigned layer, void* y,
                     void* pool_out, int N, int H, int W, void* workspace, size_t workspace_bytes,
                     unsigned int* sync, const dcb_peer_exchange_t* peers, dcb_stream_t stream);
/* dcb_bn_train_fwd with the batch sums already known (sums_q[2 C], 2^-20 fixed point, from dcb_conv*_fwd_stats): one pass
 * over the tensor, no grid barrier, any grid size.  With peers the totals of all ranks are exchanged inside the kernel as
 * above. */
int dcb_bn_train_fwd_sums(int dtype, const void* x, long long M, int C, long long M_total, const long long* sums_q,
                          const float* gamma, const float* beta, float eps, float momentum, float* moving_mean,
                          float* moving_var, float* scale, float* shift, float* mean, float* rstd, int relu, float p_drop,
                          unsigned long long seed, const unsigned long long* seed_dev, unsigned layer, void* y,
                          void* pool_out, int N, int H, int W, const dcb_peer_exchange_t* peers, dcb_stream_t stream);
int dcb_bn_train_bwd(int dtype, const float* dy, int ldy, int offy, const void* x, long long M, int C,
                     long long M_total, const float* scale, const float* shift, const float* mean,
                     const float* rstd, float p_drop, unsigned long long seed,
                     const unsigned long long* seed_dev, unsigned layer, float dgb_scale, void* draw,
                     float* dgamma, float* dbeta, void* workspace, size_t workspace_bytes, unsigned int* sync,
                     const dcb_peer_exchange_t* peers, dcb_stream_t stream);
/* the same with the upstream gradient given as the rank-1 product dy[r][c] = gpix[r] * wd[c] (dcb_head_loss_bwd_rank1): the
 * BatchNorm backward of the block in front of the softmax head never reads (and nobody writes) a materialised dL/dx */
int dcb_bn_train_bwd_rank1(int dtype, const float* gpix, const float* wd, const void* x, long long M, int C,
                           long long M_total, const float* scale, const float* shift, const float* mean,
                           const float* rstd, float p_drop, unsigned long long seed,
                           const unsigned long long* seed_dev, unsigned layer, float dgb_scale, void* draw,
                           float* dgamma, float* dbeta, void* workspace, size_t workspace_bytes, unsigned int* sync,
                           const dcb_peer_exchange_t* peers, dcb_stream_t stream);

/* ---- peer-mapped memory between the ranks of one NVSwitch box (csrc/peer.cu; SURVEY 8e, no reference counterpart:
 * the reference is single-device).  dcb_peer_alloc returns a zero-filled device buffer and its 64-byte CUDA IPC handle;
 * the other ranks map it with dcb_peer_open (the host ships the handles, e.g. with torch.distributed).  Flags are uint64
 * words in such buffers; epochs come from device-resident counters so that captured CUDA graphs stay valid. ---- */
int dcb_peer_alloc(size_t bytes, void** ptr, unsigned char* handle_out /* 64 bytes */);
int dcb_peer_open(const unsigned char* handle /* 64 bytes */, void** ptr);
int dcb_peer_close(void* ptr);
int dcb_peer_free(void* ptr);
int dcb_counter_advance(unsigned long long* counter, dcb_stream_t stream);
/* every flag_ptrs[i] (i < n <= 8; pointers may be peer-mapped) = *epoch_dev + offset, after a system-scope fence */
int dcb_flag_signal(unsigned long long* const* flag_ptrs, int n, const unsigned long long* epoch_dev, long long offset,
                    dcb_stream_t stream);
/* block the stream until flags[0..n) == *epoch_dev + offset (at_least != 0: >=); traps after ~10 s */
int dcb_flag_wait(const unsigned long long* flags, int n, const unsigned long long* epoch_dev, long long offset,
                  int at_least, dcb_stream_t stream);
/* one-shot all-reduce (sum, rank order, bit-identical on every rank) of n doubles through the peer exchange slots */
int dcb_peer_allreduce_f64(double* vals, int n, const dcb_peer_exchange_t* peers, dcb_stream_t stream);

/* Device half of the training crop sampler (unet_2d_summary.py:434-530, _batch_gen): B crops of window x window pixels.
 * img_ptrs / mask_ptrs / widths: device tables over the datasets (fp32 summary images, uint8 masks, row pitch in pixels).
 * desc: device int32 [B][12] = {dataset, y0, x0, valid rows, valid cols, m00, m01, m10, m11, t0, t1, 0}: output pixel
 * (i, j) reads window position (m00*i + m01*j + t0, m10*i + m11*j + t1) (the composed flips / rot90s), zero outside the
 * valid rows x cols.  The host keeps the reference's RNG stream and only ships these integers. */
int dcb_crop_batch(const long long* img_ptrs, const long long* mask_ptrs, const int* widths, const int* desc, int B,
                   int window, float* x_out, unsigned char* y_out, dcb_stream_t stream);
/* nearest-neighbour 2x upsampling (UpSampling2D of the `upsampling_or_transpose='upsampling'` graph, unet_2d_summary.py:160-161)
 * with the Dropout the reference applies to the upsampled tensor folded in (p_drop = 0: none): x [N][h][w][C] -> y [N][2h][2w][C];
 * backward sums the (masked) 2x2 gradient blocks of the fp32 view dy (row stride ldy, channel offset offy) into dx [N][h][w][C] */
int dcb_upsample2x(int dtype, const void* x, int N, int h, int w, int C, float p_drop, unsigned long long seed,
                   const unsigned long long* seed_dev, unsigned layer, void* y, dcb_stream_t stream);
int dcb_upsample2x_bwd(const float* dy, int ldy, int offy, int N, int h, int w, int C, float p_drop, unsigned long long seed,
                       const unsigned long long* seed_dev, unsigned layer, float* dx, dcb_stream_t stream);
/* ---- a5: MaxPooling2D(2,2) fwd and bwd (gradient to the first maximum of the window), the bwd
 * fused with the add of the skip-connection gradient (a channel slice of a concat gradient) ---- */
int dcb_maxpool2x2(int dtype, const void* x, int N, int H, int W, int C, void* y, dcb_stream_t stream);
int dcb_pool_bwd_add(int dtype, const float* skipgrad, int lds, int offs, const void* y, const void* pooled,
                     const float* dpool, int N, int H, int W, int C, float* out, dcb_stream_t stream);

/* ---- a6/a7: Conv2D(2,1,softmax)[..., -1] head (unet_2d_summary.py:221-222), losses and the
 * seven batch metrics (utils/neurons.py:13-106).  w is [C][2], b is [2] (Keras layout). ---- */
int dcb_head_fwd(int dtype, const void* x, long long M, int C, const float* w, const float* b, float* logit,
                 float* prob, dcb_stream_t stream);
/* sums[8] (double, caller zeroes): sum yt, p, yt*p, p^2, round(p), yt*round(p), BCE, weighted BCE */
int dcb_head_loss_fwd(int dtype, const void* x, long long M, int C, const float* w, const float* b,
                      const uint8_t* yt, float* prob, double* sums, dcb_stream_t stream);
/* dx[M][C] = dL/dx; dw_out[2C+2] = dL/d(kernel [C][2], bias [2]); metrics_out[8] =
 * loss, F1, prec, reca, dice, dicesq, posyt, posyp; dwb_accum[2C+2] double scratch (caller zeroes) */
int dcb_head_loss_bwd(int dtype, const void* x, long long M, int C, const float* w, const uint8_t* yt,
                      const float* prob, const double* sums, int loss, long long M_total, float* dx,
                      double* dwb_accum, float* dw_out, float* metrics_out, dcb_stream_t stream);

/* ---- a10: 8x test-time augmentation (utils/neurons.py:112-137, unet_2d_summary.py:569-595) ----
 * make_batch: reflect-pad s[hs][ws] to S x S and write transforms first..first+count-1 as [count][S][S];
 * combine: act = sum_k float32(inv_k(p_k) / n_aug) in float64, cropped to hs x ws; mask = act > threshold */
int dcb_tta_make_batch(int dtype, const float* s, int hs, int ws, int S, int first, int count, void* out,
                       dcb_stream_t stream);
int dcb_tta_combine(const float* probs, int S, int hs, int ws, float threshold, int n_aug, double* act,
                    uint8_t* mask, dcb_stream_t stream);
/* Overlap-tile TTA for images larger than the window.  The canvas is s[hs][ws] reflect-padded at the bottom and right; a
 * plan cuts it into T x T tiles with origins (origins_y[ty], origins_x[tx]) on an n_ty x n_tx grid, numbered row-major,
 * and tile (ty, tx) owns canvas rows [cuts_y[ty-1], cuts_y[ty]) and columns [cuts_x[tx-1], cuts_x[tx]) (n_ty - 1 and
 * n_tx - 1 cuts; the first and last tile own up to the canvas edge).  The plan arrays are caller-owned device int32 arrays,
 * so a captured CUDA graph keeps reading the same plan.  A call handles the group of tiles tile_first..tile_first+n_tiles-1.
 * make_batch: out [n_tiles][count][T][T] = each tile of the group under transforms first..first+count-1;
 * combine: probs [n_tiles][n_aug][T][T] -> act / mask at the image pixels the group owns (act = sum_k float32(inv_k(p_k) /
 * n_aug) in float64, mask = act > threshold); every pixel is written by exactly one group. */
int dcb_tile_make_batch(int dtype, const float* s, int hs, int ws, int T, const int* origins_y, const int* origins_x,
                        int n_ty, int n_tx, int tile_first, int n_tiles, int first, int count, void* out,
                        dcb_stream_t stream);
int dcb_tile_combine(const float* probs, int T, int hs, int ws, const int* origins_y, const int* origins_x,
                     const int* cuts_y, const int* cuts_x, int n_ty, int n_tx, int tile_first, int n_tiles, float threshold,
                     int n_aug, double* act, uint8_t* mask, dcb_stream_t stream);

/* ---- N3: Neurofinder scoring of predicted masks (datasets/nf.py:153-174: skimage.measure.label, neurofinder.centers /
 * shapes, threshold 5) and the validation windows of fit (unet_2d_summary.py:62-120); csrc/regions.cu ----
 * Images are given by a table of n_images records of 8 x int64 {data pointer, H, W, row stride, column stride, kind, 0, 0}:
 * pixel (y, x) is element y * row_stride + x * column_stride (signed, in elements), so flips, rotations and crops are views.
 * kind 0: uint8, foreground = nonzero; 1: fp32 and 2: fp64, foreground = round(p) != 0, i.e. !(|p| <= 0.5) (NaN is
 * foreground).  `desc` is the table on the device (read by the kernels), `h_desc` the same table on the host (shapes only,
 * read during the call).  H and W < 2^24, at most 2^31 - 1 pixels per call.
 * Regions are the 8-connected components numbered like scipy.ndimage.label(m != 0, structure=ones((3, 3))): in raster
 * order of their first pixel.  Regions get global numbers in table order: image i holds regions
 * [region_base[i], region_base[i+1]), region_base[n_images] = total.
 * workspace_bytes: the workspace of both calls below; region_capacity bounds the total number of regions (the rows
 * region_info must have). */
int dcb_nf_score_workspace_bytes(const long long* h_desc, int n_images, size_t* bytes, long long* region_capacity);
/* labels int32 [sum of H*W]: image i row-major at the sum of the earlier images' H*W, 1..n_i per region, 0 background */
int dcb_label_regions(const long long* desc, const long long* h_desc, int n_images, int* labels, int* region_base,
                      void* workspace, size_t workspace_bytes, dcb_stream_t stream);
/* n_pairs (truth, prediction) pairs of equal shape, as images 2p and 2p+1 of the table.  region_info int32
 * [region_capacity][3] per region = {pixel count, match, overlap}: for a truth region, match is the index (from 0) of the
 * prediction region of its pair that neurofinder.match(truth, prediction, 5) assigns to it (nearest remaining centre by
 * correctly rounded float64 distance < 5, ties to the smaller index, truth regions in label order) or -1, and overlap
 * is the number of its pixels inside that region; prediction regions carry {count, -1, 0}. */
int dcb_nf_score(const long long* desc, const long long* h_desc, int n_pairs, int* region_base, int* region_info,
                 void* workspace, size_t workspace_bytes, dcb_stream_t stream);
/* Truth mask of a dataset (unet_2d_summary.py:244-291, _summarize_mask): masks [n][H][W], one byte per pixel (int8, uint8
 * or bool; a neuron owns the pixels where its plane == 1) -> out [H][W] uint8, 1 where the reference's summary is 1.0.
 * Pixels owned by several neurons are dropped; then the survivors are visited in (owner, y, x) order and every visited
 * centre whose alive 3 x 3 window holds two owners drops that whole window.  The result is bit-identical to that
 * sequential walk: only centres whose initial window holds two owners can drop anything, and those more than 3 px apart
 * (in separate components of the dilated candidate map, labelled as in dcb_label_regions) never interact, so each
 * component is sorted and walked on its own.  n == 0 writes zeros and needs no workspace.  H and W < 2^24, H * W < 2^31. */
int dcb_mask_summary_workspace_bytes(int n, int H, int W, size_t* bytes);
int dcb_mask_summary(const uint8_t* masks, int n, int H, int W, uint8_t* out, void* workspace, size_t workspace_bytes,
                     dcb_stream_t stream);
/* out [H][W] = np.pad(f(s), ((0, H - hf), (0, W - wf)), 'reflect') for s [hs][ws] and f = (identity, np.fliplr, np.flipud,
 * np.rot90 k=1, 2, 3)[k] (hf x wf = shape of f(s); H >= hf, W >= wf) */
int dcb_orient_pad_f32(const float* s, int hs, int ws, int k, int H, int W, float* out, dcb_stream_t stream);

/* ---- a9: keras.optimizers.Adam (2.0.6) over one flat fp32 parameter buffer;
 * lr_t = lr*sqrt(1-b2^t)/(1-b1^t) is computed by the caller (unet_2d_summary.py:335) ---- */
int dcb_adam_step(float* p, const float* g, float* m, float* v, long long n, float lr_t, const float* lr_t_dev,
                  float beta1, float beta2, float eps, dcb_stream_t stream);
/* device-resident step state {iteration, dropout seed}: iteration += 1, seed advances, lr_t_out gets the
 * bias-corrected step size; dropout kernels xor *seed_dev into their seed, Adam reads *lr_t_dev
 * (both optional, NULL = use the by-value argument) so a captured CUDA graph stays valid across steps */
int dcb_step_advance(unsigned long long* state, float lr, float beta1, float beta2, float* lr_t_out,
                     dcb_stream_t stream);

int dcb_cast_from_f32(int dtype, const float* in, long long n, void* out, dcb_stream_t stream);
int dcb_cast_to_f32(int dtype, const void* in, long long n, float* out, dcb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DCB200_H_ */
