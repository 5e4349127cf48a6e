/*
 * b200seg.h — C ABI of libb200seg.so: the sm_100a kernels behind the HRNet-OCR-MScale hot path of
 * NVIDIA/semantic-segmentation (reference @ /root/reference).
 *
 * Conventions (SURVEY.md §8b "What the C-ABI replacement must export"):
 *   - plain pointers and sizes only; every buffer (including workspaces) is owned by the caller;
 *     the library never allocates, frees or retains a pointer past return;
 *   - every entry point takes the CUDA stream it must launch on (cudaStream_t passed as void*), never
 *     synchronises the device and never touches the default stream, so calls are CUDA-graph capturable;
 *   - return value: 0 = ok, negative = B200SEG_E_* argument/driver-entry error, positive = cudaError_t;
 *   - activations are NHWC ("channels-last") bf16 with an explicit pixel pitch `ld` (elements between
 *     consecutive pixels, >= channels, multiple of 8) so channel slices of a wider buffer are addressable
 *     (concat == channel offset); statistics, logits, losses are fp32; labels int64.
 *
 * Each entry point cites the reference call site (file:line under /root/reference) whose library call it replaces.
 */
#ifndef B200SEG_H_
#define B200SEG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200SEG_E_BADARG (-1)      /* shape / alignment not supported by the kernel */
#define B200SEG_E_NODRIVER (-100)  /* cuTensorMapEncodeTiled entry point unavailable */
#define B200SEG_MAX_CTAS 148       /* SMs of a B200 */
#define B200SEG_MAX_GRID 296       /* persistent grids: at most two co-resident CTAs per SM (narrow Cout tiles) */

/* ABI / build identification. */
int b200seg_abi_version(void);
const char* b200seg_build_info(void);

/* ------------------------------------------------------------------------------------------------
 * Convolution as implicit GEMM on tcgen05 (TMA-fed, TMEM accumulators).
 * Replaces cuDNN behind nn.Conv2d at network/hrnetv2.py:31-34,74-80,193-198,208-210,270-274,
 * network/ocrnet.py:54-57,66-76, network/ocr_utils.py:68-91,142-144, network/utils.py:348-362.
 * ------------------------------------------------------------------------------------------------ */
typedef struct b200seg_conv_desc {
  int32_t n, h, w;         /* INPUT batch / height / width */
  int32_t cin, cout;       /* cin multiple of 8 */
  int32_t ksize;           /* 1 or 3 (square) */
  int32_t stride;          /* 1 or 2 */
  int32_t pad;             /* 0 for 1x1, 1 for 3x3 (= dilation for dilated 3x3) */
  int32_t x_ld;            /* input pixel pitch (elements) */
  int32_t y_ld;            /* output pixel pitch (elements) */
  int32_t out_fp32;        /* 0: bf16 output, 1: fp32 output (logit heads) */
  int32_t has_bias;        /* bias[cout] fp32 added before rounding */
  int32_t emit_stats;      /* write per-CTA per-channel sum / sum-of-squares partials of the stored output */
  int32_t reserved;
  int32_t dilation;        /* 0 or 1: dense; d > 1: 3x3 taps d pixels apart, pad must equal d (WideResNet-38 mod5-7, ASPP:
                              network/wider_resnet.py:322-330, network/utils.py:176-192) */
} b200seg_conv_desc;

/* Host-only introspection of the launch plan (tests, tuning): which = 0 forward, 1 stride-1 data gradient.
 * out[10] = {kernel (1 = halo-tile 3x3, 0 = per-tap implicit GEMM), Cout tile, Cout tiles, grid, dynamic shared memory
 * bytes, ring depth, CTAs per SM, TMEM columns, resident weights, weight slots}. Returns 0 or a negative error. */
int b200seg_conv2d_plan_info(const b200seg_conv_desc* d, int32_t which, int32_t* out);

/* Diagnostics (needs a GPU): CTAs per SM the runtime grants kernel (1 = halo-tile 3x3, 0 = per-tap) in its
 * co-resident (occ_variant 2) or full-SM (1) build with smem_bytes of dynamic shared memory; negative = error. */
int32_t b200seg_debug_occupancy(int32_t kernel, int32_t occ_variant, int32_t smem_bytes);
/* prints (stdout) the device limits, the kernels' resource usage and blocks/SM as a function of dynamic shared memory */
void b200seg_debug_occupancy_report(void);

/* Process-wide planner setting: bytes of shared memory per SM every tensor-core kernel leaves unused (default 0).
 * SyncBN mode sets 12288: the one-warp kernels that wait for a peer GPU's BatchNorm statistics (1 KB of reserved shared
 * memory each) must fit on an SM next to ANY convolution CTA, otherwise a waiting warp can keep a persistent
 * convolution of another stream from completing and two GPUs wait for each other forever. */
int b200seg_set_smem_reserve(int32_t bytes);

/* Number of fp32 elements the stats partial buffer must hold: B200SEG_MAX_GRID * 2 * cout_padded. */
size_t b200seg_conv2d_stats_elems(const b200seg_conv_desc* d);

/* y[n,ho,wo,co] = sum_{kh,kw,ci} x[n, ho*s+kh-p, wo*s+kw-p, ci] * w[co,kh,kw,ci] (+ bias[co]).
 * x: bf16 NHWC (pitch x_ld); w: bf16 [cout][k*k][cin] ("OHWI", see b200seg_pack_weight); y: bf16|fp32 NHWC.
 * stats (optional): fp32 [grid][2][cout_pad]; *stats_grid receives the number of valid partial rows. */
int b200seg_conv2d_fwd(const b200seg_conv_desc* d, const void* x, const void* w_ohwi, const float* bias, void* y,
                       float* stats_partials, int32_t* stats_grid, void* stream);

/* The same convolution with the training-mode BatchNorm statistics FINALISED inside the launch (no partial table, no
 * bn_finalize launch): every CTA adds its per-channel sums to `accum` (fp64), the last CTA to finish writes
 * scale / shift / mean / invstd (and the batch statistics / running statistics exactly like b200seg_bn_finalize) and
 * clears `accum` / `counter` again. accum: [2][roundup16(cout)] fp64 and counter: uint32, both owned by the caller,
 * zero before the first use and private to one (layer, scale pass) - launches that share them must be stream ordered.
 * Per-GPU statistics only (SyncBN uses b200seg_conv2d_fwd + b200seg_bn_finalize, whose exchange needs its own kernel). */
typedef struct b200seg_bn_fold {
  double* accum;
  uint32_t* counter;
  const float* gamma;            /* may be NULL (1) */
  const float* beta;             /* may be NULL (0) */
  float* scale;
  float* shift;
  float* mean;
  float* invstd;
  float* batch_stats_out;        /* [2*c] = [mean | unbiased var] or NULL */
  float* running_mean;           /* NULL with batch_stats_out (deferred b200seg_bn_running_update) */
  float* running_var;
  int64_t* num_batches_tracked;
  float eps, momentum, count;    /* count = n * ho * wo */
  int32_t c;
} b200seg_bn_fold;
int b200seg_conv2d_fwd_bn(const b200seg_conv_desc* d, const void* x, const void* w_ohwi, const float* bias, void* y,
                          const b200seg_bn_fold* fold, void* stream);

/* Deferred variant (fold->counter == NULL; only accum and c are read): the launch adds its statistics to the cells and
 * nothing else - the BatchNorm apply pass that consumes the layer finalises them in its prologue (b200seg_bn_apply_cells),
 * so no finaliser launch and no last-CTA tail sits between the convolution and its consumer. The caller zeroes the cells
 * once per step. */

/* The same with a residual addend: y = conv(x) (+ bias) + addend[n,ho,wo,cout] (bf16, pitch addend_ld); the statistics
 * are those of the stored sum (pre-activation residual networks: network/wider_resnet.py:170-183). bf16 output only. */
int b200seg_conv2d_fwd_add(const b200seg_conv_desc* d, const void* x, const void* w_ohwi, const float* bias,
                           const void* addend, int32_t addend_ld, void* y, float* stats_partials, int32_t* stats_grid,
                           void* stream);

/* Evaluation mode: BatchNorm from running statistics, the residual sum and the ReLU folded into the convolution epilogue:
 *   y = relu?(conv(x) * scale[co] + shift[co] (+ addend[n,ho,wo,co]))      (network/hrnetv2.py:50-66,86-106 in one launch)
 * scale / shift: fp32 [cout] (b200seg_bn_eval_params; a convolution bias is folded into shift by the caller), bf16 output,
 * d->has_bias = d->emit_stats = d->out_fp32 = 0. */
int b200seg_conv2d_fwd_affine(const b200seg_conv_desc* d, const void* x, const void* w_ohwi, const float* scale,
                              const float* shift, int32_t relu, const void* addend, int32_t addend_ld, void* y,
                              void* stream);

/* Repack fp32 OIHW master weights (the nn.Parameter layout the reference checkpoints use) into the kernel layouts:
 *   w_ohwi  bf16 [O][kh*kw][I]            forward operand
 *   w_dgrad bf16 [I][kh*kw (flipped)][o_pad]  data-gradient operand (may be NULL); o_pad >= O is a multiple of 8 and
 *           the pad columns must have been zeroed by the caller once (they are never written). */
int b200seg_pack_weight(const float* w_oihw, int32_t o, int32_t i, int32_t ksize, void* w_ohwi, void* w_dgrad,
                        int32_t o_pad, void* stream);

/* The same repack for every convolution of the model in one launch (the weights change every optimizer step).
 * items: DEVICE array; block b handles b200seg_pack_chunk() consecutive OIHW elements of items[blk_item[b]] starting
 * at blk_start[b]. i_dst >= i is the input-channel extent of the destination layouts (the 3-channel stem runs on a
 * 16-channel padded image; pad entries must have been zeroed once by the caller). which: 1 = forward operands only,
 * 2 = data-gradient operands only (needed from the backward on: can run on a side stream), 3 = both. */
typedef struct b200seg_pack_item {
  const void* w_oihw;      /* fp32 [o][i][k][k] */
  void* w_ohwi;            /* bf16 [o][k*k][i_dst] or NULL */
  void* w_dgrad;           /* bf16 [i_dst][k*k flipped][o_pad] or NULL */
  int32_t o, i, i_dst, ksize, o_pad, reserved;
} b200seg_pack_item;
int32_t b200seg_pack_chunk(void);
int b200seg_pack_weights(const b200seg_pack_item* items, const int32_t* blk_item, const int32_t* blk_start,
                         int32_t n_blocks, int32_t which, void* stream);

/* Data gradient: dx[n,h,w,cin] = conv_transpose(dy, W) (+ addend, e.g. a gradient that already arrived at x).
 * d describes the FORWARD convolution; dy: bf16 [n,ho,wo,*] whose channel extent is roundup8(cout) (pad channels
 * zero); w_dgrad from b200seg_pack_weight with o_pad = roundup8(cout). Stride-2 convolutions run as four parity-class
 * launches of the same tcgen05 kernel. Replaces cuDNN convolution_backward (input part). */
int b200seg_conv2d_dgrad(const b200seg_conv_desc* d, const void* dy, int32_t dy_ld, const void* w_dgrad,
                         const void* addend, int32_t addend_ld, void* dx, int32_t dx_ld, void* stream);


/* Weight gradient: dw_ohwi[co][kh*kw][ci] (fp32 accumulator in the kernels' own layout, 16-byte aligned)
 *   += sum_pixels dy[.., co] * x_shifted[.., ci]        (the convolution weight gradient, SURVEY.md K1-K5).
 * d describes the FORWARD convolution (input geometry, stride, pad); dy is bf16 NHWC [n,ho,wo,cout] with pitch dy_ld;
 * cin multiple of 16. Deterministic. Depending on the shape the tcgen05 kernel either owns every gradient element
 * (one launch, no workspace) or writes per-work-unit fp32 slabs into the caller's workspace that a second kernel sums
 * in a fixed order; _ws_bytes / _launches report which. b200seg_grad_fold turns the accumulators into OIHW gradients. */
size_t b200seg_conv2d_wgrad_ws_bytes(const b200seg_conv_desc* d);
int32_t b200seg_conv2d_wgrad_launches(const b200seg_conv_desc* d);
int b200seg_conv2d_wgrad(const b200seg_conv_desc* d, const void* x, const void* dy, int32_t dy_ld, float* dw_ohwi,
                         void* workspace, size_t ws_bytes, void* stream);

/* End-of-step gradient fold: dst and the two accumulators share ONE flat fp32 layout (element offsets in segs):
 *   conv weights: dst[co][ci][tap] (OIHW, the nn.Parameter .grad layout) (+)= acc_a[co][tap][ci'] + acc_b[co][tap][ci']
 *                 with ci' running over src_cin >= cin input channels of the accumulator (the stem accumulates on the
 *                 16-channel padded image: src_cin = 16, cin = 3) starting at src_offset;
 *   vectors (BN affine, biases; cout = 1, taps = 1, cin = numel): dst[i] (+)= acc_a[i] + acc_b[i].
 * mode bit 0 (clear): zero what was read from acc_a / acc_b; bit 1 (overwrite): dst = sum instead of dst += sum (dst is
 * then not read). Either accumulator may be NULL. One thread block per chunk of b200seg_grad_fold_chunk() consecutive
 * elements of one segment: blk_seg[b] indexes segs, blk_start[b] is the first element of the chunk inside its segment.
 * Replaces autograd's gradient accumulation across the two scale passes (network/ocrnet.py:278-281). */
typedef struct b200seg_grad_seg {
  int64_t offset;          /* first element of the parameter in dst */
  int64_t src_offset;      /* first element of its accumulator in acc_a / acc_b */
  int32_t cout, cin, taps; /* conv: [cout][cin][taps]; vector: cout = 1, cin = numel, taps = 1 */
  int32_t src_cin;         /* input channels per tap in the accumulator (>= cin) */
} b200seg_grad_seg;
int32_t b200seg_grad_fold_chunk(void);
int b200seg_grad_fold(float* dst, float* acc_a, float* acc_b, const b200seg_grad_seg* segs, const int32_t* blk_seg,
                      const int32_t* blk_start, int32_t n_blocks, int32_t mode, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Training-mode BatchNorm around the convolutions. Replaces cuDNN/Apex BN behind Norm2d (network/mynn.py:18-24),
 * in-place ReLU (network/hrnetv2.py:28,44) and the residual add (network/hrnetv2.py:63-64,103-104).
 * ------------------------------------------------------------------------------------------------ */
/* SyncBN (apex.parallel.SyncBatchNorm behind Norm2d, config.py:216-225; collective C2 of SURVEY.md §2b): optional
 * cross-GPU exchange fused into the two finalisers. Every rank owns a mailbox (fp64) and a flag array (uint32) that all
 * peers of the node can write through NVLink (b200seg_p2p_*). NULL or world <= 1: per-GPU statistics.
 *   mail layout : [parity 2][exchange][rank][2][c] doubles  (parity = step & 1, parity_stride doubles per half)
 *   flag layout : [exchange][rank][ceil(c/32)] uint32, written with the step number (release), polled (acquire)
 * Every rank must issue the same sequence of exchanges with the same offsets; *step is read on the device and must be
 * incremented by the caller once per training step (inside the captured graph). */
typedef struct b200seg_bn_sync {
  const void* mail_peers;   /* device array [world] of double*: mailbox base of every rank as mapped on this rank */
  const void* flag_peers;   /* device array [world] of uint32_t*: flag base of every rank as mapped on this rank */
  const void* step;         /* device uint32_t* step counter */
  int64_t mail_offset;      /* offset of this exchange inside a parity half, in doubles */
  int64_t parity_stride;    /* doubles per parity half */
  int32_t flag_offset;      /* offset of this exchange in the flag array */
  int32_t world, rank;
  int32_t reserved;
  void* beacon;             /* optional host-mapped int32[8] post-mortem record: [0,1] = (flag_offset, step) of the last
                               exchange this rank entered, [4,5] = of the last one it completed; NULL = off */
} b200seg_bn_sync;
/* Peer-mappable device memory for the SyncBN mailboxes: the ONLY allocations the library performs (a communicator
 * owns its buffers). alloc: cudaMalloc + zero + CUDA IPC handle (64 bytes) to hand to the other ranks of the node;
 * open: map a peer's buffer (lazy peer access over NVLink); close / free release them. */
int b200seg_p2p_alloc(size_t bytes, void** dev_ptr, uint8_t* handle64);
int b200seg_p2p_open(const uint8_t* handle64, void** dev_ptr);
int b200seg_p2p_close(void* dev_ptr);
int b200seg_p2p_free(void* dev_ptr);

/* partials[grid][2][cpad] (conv epilogue) -> scale = gamma*invstd, shift = beta - mean*scale, saved mean/invstd;
 * running stats updated with `momentum` (unbiased variance), num_batches_tracked += 1 (all optional);
 * batch_stats_out (optional) receives [mean c | unbiased var c] for a deferred b200seg_bn_running_update. */
int b200seg_bn_finalize(const float* partials, int32_t grid, int32_t c, int32_t cpad, float count, const float* gamma,
                        const float* beta, float eps, float momentum, float* running_mean, float* running_var,
                        int64_t* num_batches_tracked, float* scale, float* shift, float* mean, float* invstd,
                        float* batch_stats_out, const b200seg_bn_sync* sync, void* stream);
/* Momentum update of every BatchNorm layer's running statistics in one launch: running / batch_pass* are flat fp32
 * buffers of n elements with one layout ([mean c | var c] per layer); pass 0 is applied before pass 1 (the order of
 * the two _fwd calls in network/ocrnet.py:278-281); batch_pass1 may be NULL. num_batches_tracked[n_layers] += n_passes
 * (the BatchNorm2d bookkeeping behind Norm2d, network/mynn.py:18-24). */
int b200seg_bn_running_update(float* running, const float* batch_pass0, const float* batch_pass1, int64_t n,
                              float momentum, int64_t* num_batches_tracked, int32_t n_layers, int32_t n_passes,
                              void* stream);
/* Multi-tensor SGD step (the update rule of the optimizer loss/optimizer.py:43-60 builds: momentum, weight decay,
 * optional nesterov) for every parameter of a group in ONE launch. items: DEVICE array; block b updates
 * b200seg_sgd_chunk() consecutive elements of items[blk_item[b]] from blk_start[b]. first_step: momentum buffers are
 * initialised with the (decayed) gradient. SURVEY.md §8(f) row f3. */
typedef struct b200seg_sgd_item {
  void* param;             /* fp32 [numel] */
  const void* grad;        /* fp32 [numel] */
  void* momentum_buf;      /* fp32 [numel] (ignored when momentum == 0) */
  int64_t numel;
} b200seg_sgd_item;
int32_t b200seg_sgd_chunk(void);
int b200seg_sgd_step(const b200seg_sgd_item* items, const int32_t* blk_item, const int32_t* blk_start, int32_t n_blocks,
                     float lr, float momentum, float dampening, float weight_decay, int32_t nesterov, int32_t first_step,
                     void* stream);

/* dst[n] += src[n] (fp32, n multiple of 4, 16-byte aligned): folds a scale pass' private parameter-gradient buffer
 * into the step gradient (the passes run concurrently; autograd's accumulation order lo -> hi is kept). */
int b200seg_accum_f32(float* dst, const float* src, int64_t n, void* stream);
/* Gradient publish (the step's autograd boundary): dst = (accumulate ? dst : 0) + (*scale_dev * scale_const) * src over n
 * fp32 elements (n multiple of 4, 16-byte aligned). scale_dev (device pointer, may be NULL = 1) is the upstream gradient
 * of the loss handed to backward() - amp.scale_loss / loss / accumulation_steps (train.py:499-505) - scale_const the
 * 1 / world_size of the data-parallel average (network/__init__.py:38-39 apex DDP). */
int b200seg_publish_grads(float* dst, const float* src, int64_t n, const float* scale_dev, float scale_const,
                          int32_t accumulate, void* stream);
/* eval mode: scale/shift from running statistics */
int b200seg_bn_eval_params(int32_t c, const float* gamma, const float* beta, float eps, const float* running_mean,
                           const float* running_var, float* scale, float* shift, void* stream);
/* z = relu?(y*scale + shift [+ res]) [* post_scale[n][c]]   (post_scale carries the Dropout2d mask/(1-p),
 * network/ocr_utils.py:146). npix = n*h*w, hw = h*w. */
int b200seg_bn_apply(const void* y, int32_t y_ld, const float* scale, const float* shift, const void* res,
                     int32_t res_ld, const float* post_scale, int32_t relu, void* z, int32_t z_ld, int64_t npix,
                     int32_t hw, int32_t c, void* stream);
/* The same pass as the consumer of a convolution launched in deferred mode (b200seg_conv2d_fwd_bn with counter == NULL):
 * every block derives scale / shift from f->accum (fp64 [2][roundup16(c)] sums), block 0 writes f->scale / shift / mean /
 * invstd (+ batch or running statistics exactly like b200seg_bn_finalize). f->counter is ignored. */
int b200seg_bn_apply_cells(const void* y, int32_t y_ld, const b200seg_bn_fold* f, const void* res, int32_t res_ld,
                           const float* post_scale, int32_t relu, void* z, int32_t z_ld, int64_t npix, int32_t hw,
                           int32_t c, void* stream);
/* backward: g = dz * post_scale * (mask > 0); partials[grid][2][c] of (sum g, sum g*xhat), grid from _bn_bwd_grid */
int32_t b200seg_bn_bwd_grid(int64_t npix, int32_t c);
int b200seg_bn_bwd_reduce(const void* dz, int32_t dz_ld, const void* mask, int32_t mask_ld, const float* post_scale,
                          const void* y, int32_t y_ld, const float* mean, const float* invstd, int64_t npix, int32_t hw,
                          int32_t c, float* partials, void* stream);
/* dgamma += sum g*xhat, dbeta += sum g (accumulating), c1 = sum g / count, c2 = sum g*xhat / count */
int b200seg_bn_bwd_finalize(const float* partials, int32_t grid, int32_t c, float count, float* dgamma, float* dbeta,
                            float* c1, float* c2, const b200seg_bn_sync* sync, void* stream);
/* bn_bwd_reduce with the finalisation folded into the launch (per-GPU statistics; csrc/bn_fold.cuh pattern): CTAs add
 * their sums to accum ([2][c] fp64, zero between launches, private to one layer and scale pass), the last CTA adds
 * dgamma / dbeta, writes c1 = sum(g)/npix, c2 = sum(g*xhat)/npix and clears accum / counter. */
int b200seg_bn_bwd_reduce_finalize(const void* dz, int32_t dz_ld, const void* mask, int32_t mask_ld,
                                   const float* post_scale, const void* y, int32_t y_ld, const float* mean,
                                   const float* invstd, int64_t npix, int32_t hw, int32_t c, double* accum,
                                   uint32_t* counter, float* dgamma, float* dbeta, float* c1, float* c2, void* stream);
/* dy = gamma*invstd*(g - c1 - xhat*c2); optionally g_out (=|+=) g for the residual / identity branch */
int b200seg_bn_bwd_apply(const void* dz, int32_t dz_ld, const void* mask, int32_t mask_ld, const float* post_scale,
                         const void* y, int32_t y_ld, const float* mean, const float* invstd, const float* gamma,
                         const float* c1, const float* c2, void* dy, int32_t dy_ld, void* g_out, int32_t g_ld,
                         int32_t g_accumulate, int64_t npix, int32_t hw, int32_t c, void* stream);
/* reduce + gradient pass with deferred finalisation (two launches): the reduction adds its sums to cells ([2][c] fp64,
 * zeroed by the caller once per step), the gradient pass folds them in its prologue and accumulates dgamma / dbeta
 * (either may be NULL). Per-GPU statistics only (SyncBN: _reduce + _finalize + _apply). */
int b200seg_bn_bwd_cells(const void* dz, int32_t dz_ld, const void* mask, int32_t mask_ld, const float* post_scale,
                         const void* y, int32_t y_ld, const float* mean, const float* invstd, const float* gamma,
                         float* dgamma, float* dbeta, double* cells, void* dy, int32_t dy_ld, void* g_out, int32_t g_ld,
                         int32_t g_accumulate, int64_t npix, int32_t hw, int32_t c, void* stream);
/* dst (=|+=) src * (mask > 0) */
int b200seg_masked_accum(const void* src, int32_t src_ld, const void* mask, int32_t mask_ld, void* dst, int32_t dst_ld,
                         int32_t accumulate, int64_t npix, int32_t c, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Multi-resolution fuse / upsample+concat / their adjoint / image preparation.
 * Replaces F.interpolate + add + ReLU chains at network/hrnetv2.py:230-254,438-447 and ResizeX (network/mynn.py:102-114).
 * ------------------------------------------------------------------------------------------------ */
typedef struct b200seg_fuse_term {
  const void* x;        /* bf16 NHWC [n, h, w, c] */
  const float* scale;   /* optional per-channel affine (BN folded), both or neither */
  const float* shift;
  int32_t ld, h, w;
  int32_t reserved;
} b200seg_fuse_term;
typedef struct b200seg_fuse_desc {
  b200seg_fuse_term term[4];
  int32_t nterms;
  int32_t n, h, w, c;   /* output geometry */
  int32_t relu;
  int32_t reserved[2];
} b200seg_fuse_desc;
/* out[n,Y,X,:] = relu?( sum_j affine_j( bilinear_j(x_j)[Y,X,:] ) ), summed in term order */
int b200seg_fuse_fwd(const b200seg_fuse_desc* d, void* out, int32_t out_ld, void* stream);
/* out[n,y,x,:] (=|+=) sum_{Y,X} w(Y,y) w(X,x) g[n,Y,X,:] * (mask>0): adjoint of the align_corners=False bilinear upsample */
int b200seg_upsample_adjoint(const void* g, int32_t g_ld, const void* mask, int32_t mask_ld, int32_t n, int32_t H,
                             int32_t W, int32_t c, void* out, int32_t out_ld, int32_t h, int32_t w, int32_t accumulate,
                             void* stream);
/* fp32 NCHW [n,3,H,W] -> bf16 NHWC [n,h,w,16] (zero padded channels), bilinear resize to (h,w) */
int b200seg_image_prep(const float* img_nchw, int32_t n, int32_t H, int32_t W, void* out_nhwc16, int32_t h, int32_t w,
                       void* stream);

/* ------------------------------------------------------------------------------------------------
 * OCR glue: softmaxes around the skinny GEMMs of SpatialGather (network/ocr_utils.py:34-46) and
 * ObjectAttentionBlock (network/ocr_utils.py:95-119). The GEMMs themselves run on b200seg_conv2d_fwd /
 * b200seg_conv2d_wgrad with the class dimension padded to a 32-wide bf16 operand.
 * ------------------------------------------------------------------------------------------------ */
int32_t b200seg_spatial_softmax_blocks(int32_t P);   /* partial_ws needs n * blocks * 32 * 2 floats */
/* probs[n][pix][k<32] = softmax over the P pixels of logits[n][pix][k] (fp32, pitch ld); k >= K -> 0 */
int b200seg_spatial_softmax_fwd(const float* logits, int32_t ld, int32_t n, int32_t P, int32_t K, float* partial_ws,
                                void* probs_bf16, float* stat_out, void* stream);
/* dlogit[n][pix][k<32] (bf16, =|+=) probs * (dprobs - sum_pix probs*dprobs) */
int b200seg_spatial_softmax_bwd(const float* dprobs, int32_t ldd, const void* probs_bf16, int32_t n, int32_t P, int32_t K,
                                float* partial_ws, void* dlogit_bf16, int32_t accumulate, void* stream);
/* sim[pix][k<32] = softmax_k(scale * x[pix][k]); ds = scale * sim * (dsim - <sim, dsim>) */
int b200seg_class_softmax_fwd(const float* x, int32_t ld, int64_t P, int32_t K, float scale, void* sim_bf16, void* stream);
int b200seg_class_softmax_bwd(const float* dsim, int32_t ld, const void* sim_bf16, int64_t P, int32_t K, float scale,
                              void* ds_bf16, void* stream);
/* dst[c][r] (bf16, pitch rpad, zero padded) = src[r][c]; src is bf16 or fp32 with pitch ld */
int b200seg_transpose_pad(const void* src, int32_t src_fp32, int32_t R, int32_t C, int32_t ld, void* dst_bf16, int32_t rpad,
                          void* stream);
/* dst bf16 [rows][dst_ld] (=|+=) src fp32 [rows][src_ld], first C columns */
int b200seg_cast_rows(const float* src, int32_t src_ld, void* dst_bf16, int32_t dst_ld, int64_t rows, int32_t C,
                      int32_t accumulate, void* stream);

/* db[c] += sum_rows dy[row][c], c < C <= 32 (bias gradient of the logit heads, network/ocrnet.py:66-76). partials is an
 * fp32 workspace of b200seg_bias_grad_blocks(rows) * 32 floats: the per-block sums are added in a fixed order (no
 * atomics), so the result does not depend on the order in which blocks finish. Two launches. */
int32_t b200seg_bias_grad_blocks(int64_t rows);
int b200seg_bias_grad(const void* dy_bf16, int32_t ld, int64_t rows, int32_t C, float* partials, float* db, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Multi-scale attention blend + cross-entropy, forward and backward (network/ocrnet.py:170-183,264-319,
 * network/mscale.py:182-220, loss/utils.py:133-134). Logit maps are fp32 [n][h][w][20] (19 classes + 1 pad),
 * class-gradient outputs bf16 [pixels][32] (zero padded) ready for b200seg_conv2d_dgrad/_wgrad.
 * ------------------------------------------------------------------------------------------------ */
typedef struct b200seg_mscale_desc {
  int32_t n, h, w;          /* labels / full resolution */
  int32_t hq, wq;           /* hi-pass quarter-resolution maps */
  int32_t hm, wm;           /* mid grid = lo-pass input size (0,0: single-scale, no lo pass) */
  int32_t hl, wl;           /* lo-pass quarter-resolution maps */
  int32_t nheads;           /* 1: cls only, 2: cls + aux */
  float w_head0, w_head1;   /* loss weights (1.0, cfg.LOSS.OCR_ALPHA) */
  float sup_wt;             /* cfg.LOSS.SUPERVISED_MSCALE_WT (0 disables) */
  int32_t ignore_index;     /* 255 */
  int32_t loss_kind;        /* 0: CrossEntropyLoss2d heads (loss/utils.py:133-134); 1: RMILoss criterion (loss/rmi.py) */
  int32_t reserved;
} b200seg_mscale_desc;
/* counter_ws: one uint64; inv_count <- 1 / (#(labels != ignore) + plus_one)   (plus_one: RMILoss normalisation) */
int b200seg_count_valid(const int64_t* labels, int64_t total, int32_t ignore_index, int32_t plus_one,
                        uint64_t* counter_ws, float* inv_count, void* stream);
/* mid[n][hm][wm][40] fp32 (attn4*cls4, attn4*aux4, attn4, 0); mid_sup[n][hm][wm][20] = cls4 when sup_wt != 0 */
int b200seg_mscale_mid_fwd(const b200seg_mscale_desc* d, const float* lo_cls, const float* lo_aux,
                           const float* lo_attn_logit, float* mid, float* mid_sup, void* stream);
int32_t b200seg_mscale_loss_blocks(const b200seg_mscale_desc* d);   /* partial_ws: blocks * 4 floats */
/* loss_out (8 floats): [0] total loss, [1..4] mean pointwise loss of {cls, aux, supervised lo, supervised hi},
 * [5] the RMI term; g_hi / g_lo / g_sup: bf16 [n*h*w][40] per-pixel gradients consumed by the backward entry points.
 * loss_kind 1 (RMILoss criterion): the pointwise loss is sigmoid BCE; rmi_dpr (fp32 [n][h/4+1][w/4+1][20], from
 * b200seg_rmi_grad) is the RMI gradient w.r.t. the pooled probabilities of head 0 and rmi_terms[n_rmi_terms] the
 * already weighted RMI values summed into the total (both NULL / 0 otherwise). */
int b200seg_mscale_loss_fwd(const b200seg_mscale_desc* d, const int64_t* labels, const float* inv_count,
                            const float* hi_cls, const float* hi_aux, const float* mid, const float* mid_sup, void* g_hi,
                            void* g_lo, void* g_sup, float* partial_ws, float* loss_out, const float* rmi_dpr,
                            const float* rmi_terms, int32_t n_rmi_terms, void* stream);
int b200seg_mscale_hi_bwd(const b200seg_mscale_desc* d, const void* g_hi, void* d_cls, void* d_aux, void* stream);
/* dmid_ws: fp32 [n*hm*wm][40]; d_attn: bf16 [n*hl*wl][8] gradient w.r.t. the PRE-sigmoid attention logit */
int b200seg_mscale_lo_bwd(const b200seg_mscale_desc* d, const void* g_lo, const void* g_sup, const float* lo_cls,
                          const float* lo_aux, const float* lo_attn_logit, const float* mid, float* dmid_ws, void* d_cls,
                          void* d_aux, void* d_attn, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Region Mutual Information head of the RMILoss criterion (loss/rmi.py:70-215, loss/rmi_utils.py:15-56,95-107) on the
 * blended logits of head 0: radius 3, avg-pool 4/4/pad 2, sigmoid probabilities, fp64 covariances, lambda 0.5.
 * Used with b200seg_mscale_desc.loss_kind = 1; the pointwise BCE part lives in b200seg_mscale_loss_fwd.
 * ------------------------------------------------------------------------------------------------ */
/* pr_pool / la_pool: fp32 [n][h/4+1][w/4+1][20] = avg_pool2d(sigmoid(joint)*mask + 1e-6) / avg_pool2d(onehot*mask) */
int b200seg_rmi_pool(const b200seg_mscale_desc* d, const int64_t* labels, const float* hi_cls, const float* mid,
                     float* pr_pool, float* la_pool, void* stream);
size_t b200seg_rmi_ws_bytes(int32_t n);
/* Second moments (fp64) -> per (image, class) 9x9 Cholesky solves -> rmi_terms[n*19] (each already multiplied by
 * scale = w_head0 * (1 - lambda) / (n * 9)) and dpr = d(sum rmi_terms) / d pr_pool, fp32 [n][h/4+1][w/4+1][20].
 * G: fp64 scratch [n][19][180]; ws: b200seg_rmi_ws_bytes(n) bytes, 8-byte aligned. Three launches. */
int b200seg_rmi_solve_grad(int32_t n, int32_t h, int32_t w, const float* pr_pool, const float* la_pool, float scale,
                           void* ws, size_t ws_bytes, double* G, float* rmi_terms, float* dpr, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Eval-mode output assembly: full-resolution fp32 NCHW maps and the hierarchical blend of
 * MscaleOCR.nscale_forward / two_scale_forward (network/ocrnet.py:185-262,289-327), mynn.Upsample / scale_as.
 * ------------------------------------------------------------------------------------------------ */
/* NHWC fp32 [n,h,w,ld] (first c channels) -> NCHW fp32 [n,c,H,W], bilinear align_corners=False; optional sigmoid first */
int b200seg_resize_to_nchw(const float* src_nhwc, int32_t ld, int32_t n, int32_t h, int32_t w, int32_t c,
                           int32_t apply_sigmoid, float* dst_nchw, int32_t H, int32_t W, void* stream);
/* NCHW fp32 [planes,h,w] -> [planes,H,W] bilinear */
int b200seg_resize_nchw(const float* src, int32_t planes, int32_t h, int32_t w, float* dst, int32_t H, int32_t W,
                        void* stream);
/* a: [n,1,hw]; mode 0: out = a*x + (1-a)*y; 1: out = x + (1-a)*y; 2: out = a*x   (x, y, out: [n,c,hw]) */
int b200seg_blend(const float* a, const float* x, const float* y, float* out, int32_t n, int32_t c, int64_t hw,
                  int32_t mode, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Pooling / broadcast glue of the DeepLabV3+ / WideResNet-38 path (SURVEY.md §8(f) f2): NHWC bf16.
 * ------------------------------------------------------------------------------------------------ */
/* nn.MaxPool2d(3, stride=2, padding=1) (network/wider_resnet.py:347-349); y: [n, (h-1)/2+1, (w-1)/2+1, c] */
int b200seg_maxpool3x3s2_fwd(const void* x, int32_t x_ld, int32_t n, int32_t h, int32_t w, int32_t c, void* y,
                             int32_t y_ld, void* stream);
/* dx (=|+=) adjoint of the above; x is the forward input (the argmax is recomputed, first maximum wins) */
int b200seg_maxpool3x3s2_bwd(const void* x, int32_t x_ld, const void* dy, int32_t dy_ld, int32_t n, int32_t h, int32_t w,
                             int32_t c, void* dx, int32_t dx_ld, int32_t accumulate, void* stream);
/* per-channel sum / sum of squares of an activation: partials fp32 [grid][2][c], grid = _channel_stats_grid(npix, c);
 * same layout as the convolution epilogues' statistics (feed b200seg_bn_finalize with cpad = c) */
int32_t b200seg_channel_stats_grid(int64_t npix, int32_t c);
int b200seg_channel_stats(const void* x, int32_t x_ld, int64_t npix, int32_t c, float* partials, void* stream);
/* out[n][c] (bf16, pitch out_ld, =|+=) scale * sum over the p pixels of x[n][pix][c]  (nn.AdaptiveAvgPool2d(1) with
 * scale = 1/p, network/utils.py:194-210; adjoint of the broadcast below with scale = 1); ws: fp32 [n][splits(p)][c] */
int32_t b200seg_spatial_sum_splits(int32_t p);
int b200seg_spatial_sum(const void* x, int32_t x_ld, int32_t n, int32_t p, int32_t c, float scale, float* ws, void* out,
                        int32_t out_ld, int32_t accumulate, void* stream);
/* out[n][pix][c] (=|+=) scale * v[n][c]: Upsample of a 1x1 map; adjoint of the image pooling with scale = 1/p */
int b200seg_broadcast_pixels(const void* v, int32_t v_ld, int32_t n, int32_t p, int32_t c, float scale, void* out,
                             int32_t out_ld, int32_t accumulate, void* stream);

/* Evaluation tail on the device (utils/trnval_utils.py:116-196 eval_minibatch, utils/misc.py:50-85 fast_hist):
 * out (=|+=) pred [n,c,h,w] fp32, optionally mirrored along w (the do_flip / multi-scale averaging loop) */
int b200seg_accum_pred(const float* pred, float* out, int32_t n, int32_t c, int32_t h, int32_t w, int32_t flip,
                       int32_t accumulate, void* stream);
/* per pixel of pred*scale [n,c,hw]: argmax class (int64, first maximum), softmax max probability (fp32) and the
 * confusion histogram hist[gt*c + pred] += 1 (int64, caller-zeroed, accumulates) over pixels with 0 <= gt < c.
 * Every output is optional (NULL); hist needs labels. */
int b200seg_argmax_hist(const float* pred_nchw, int32_t n, int32_t c, int64_t hw, float scale, const int64_t* labels,
                        int64_t* pred_out, float* maxprob_out, int64_t* hist, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Training input pipeline on the device (SURVEY.md 8 row f4): the reference's per-sample transform chain
 * (datasets/__init__.py:72-108) on the decoded uint8 frame, bit-exact with Pillow. Host side: b200seg/augment.py.
 * ------------------------------------------------------------------------------------------------ */
typedef struct b200seg_aug_geom {
  int32_t src_h, src_w;        /* decoded frame: rgb uint8 [src_h][src_w][3], label ids uint8 [src_h][src_w] */
  int32_t out_h, out_w;        /* crop size */
  int32_t win_y0, win_x0;      /* first crop row / column (before the flip) that shows a pixel of the resized frame */
  int32_t n_y, n_x;            /* rows / columns of that window = extents of the tables (0: the crop is all padding) */
  int32_t ksize_v, ksize_h;    /* row pitch of kk_v / kk_h */
  int32_t flip;                /* RandomHorizontallyFlip (transforms/joint_transforms.py:276-281) */
  int32_t ignore_label;        /* label of the padding (RandomCrop, :171-176) */
} b200seg_aug_geom;
/* RandomSizeAndCrop + RandomCrop padding + flip. kk_* int32 [n][ksize] / bounds_* int32 [n][2]: Pillow's BICUBIC taps of the
 * window's output positions (22-bit fixed point; first source index, tap count); near_* int32 [n]: NEAREST source index;
 * id_lut uint8 [256] or NULL (datasets/base_loader.py:177-181). out_rgb uint8 [out_h][out_w][3], out_label int64. */
int b200seg_aug_resize_crop(const b200seg_aug_geom* d, const uint8_t* src_rgb, const uint8_t* src_mask,
                            const int32_t* kk_h, const int32_t* bounds_h, const int32_t* kk_v, const int32_t* bounds_v,
                            const int32_t* near_x, const int32_t* near_y, const uint8_t* id_lut, uint8_t* out_rgb,
                            int64_t* out_label, void* stream);
typedef struct b200seg_aug_color {
  int32_t n_ops;               /* 0..4 ColorJitter ops in their drawn order (transforms/transforms.py:326-348) */
  int32_t kind[4];             /* 0 brightness, 1 contrast, 2 saturation, 3 hue */
  float factor[4];             /* ImageEnhance factor of ops 0-2 */
  int32_t hue_shift[4];        /* np.uint8(hue_factor * 255) of the hue op */
  float mean[3], std[3];       /* Normalize (config.py:96-97) */
} b200seg_aug_color;
/* ColorJitter -> ToTensor -> Normalize: rgb uint8 [h][w][3] -> fp32 [3][h][w]. luma_sum_ws: 8 bytes of device memory
 * (needed when a contrast op is present: ImageEnhance.Contrast blends with the mean grey level). */
int b200seg_aug_color_normalize(const b200seg_aug_color* c, const uint8_t* rgb, int32_t h, int32_t w,
                                uint64_t* luma_sum_ws, float* out_chw, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200SEG_H_ */
