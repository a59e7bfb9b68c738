/* pf_b200.h — C ABI of libpf_b200.so: the B200 (sm_100a) kernels behind PocketFlow's
 * compression-aware training step.
 *
 * The reference (Tencent/PocketFlow) has no FFI: its de-facto operator boundary is the set of
 * private learner methods that emit TensorFlow op chains.  Each entry point below replaces one
 * such chain; the comment above it cites the reference file:line it stands in for.
 *
 * Conventions (SURVEY.md §8b):
 *   - every function returns int: 0 = ok, <0 = pf_status, >0 = cudaError_t;
 *     pf_last_error() returns a thread-local human-readable message for the last failure.
 *   - the caller owns every buffer (inputs, outputs, workspaces, descriptor tables); kernels
 *     never allocate.  Pointers named *_dev are device pointers; `stream` is a cudaStream_t
 *     passed as void* (0 = legacy default stream).
 *   - all calls are asynchronous with respect to the host (enqueue only) unless stated.
 *   - fp32 everywhere ("u32"/"u8" where noted); tensors are dense, NHWC activations,
 *     HWIO ([kh,kw,cin,cout]) kernels — the TF layouts the reference uses.
 *   - there is NO CPU fallback anywhere in this library.
 */
#ifndef PF_B200_H_
#define PF_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PF_B200_ABI_VERSION 1

typedef enum pf_status {
  PF_OK = 0,
  PF_ERR_INVALID_ARG = -1,  /* bad size / null pointer / unsupported mode (Python raises ValueError) */
  PF_ERR_UNSUPPORTED = -2,  /* shape outside what the kernel implements                              */
  PF_ERR_NO_DEVICE = -3,    /* no CUDA device / driver                                              */
  PF_ERR_NCCL = -4,         /* NCCL missing or returned an error                                    */
  PF_ERR_INTERNAL = -5
} pf_status;

int pf_abi_version(void);
const char* pf_last_error(void);
/* Number of kernel launches this library has enqueued in this process (bench.py "gpu_launches"). */
int64_t pf_launch_count(void);
void pf_launch_count_reset(void);
/* Device query helper: SM count of the current device (148 on B200). */
int pf_sm_count(int* out);

/* ---------------------------------------------------------------------------------------------
 * Ordered-uint encoding of float min/max slots.  enc(f) is monotone in f, so atomicMin/atomicMax
 * on uint32 implement float min/max.  A min slot starts at 0xFFFFFFFF, a max slot at 0.
 *   enc(f) = bits(f) ^ (bits(f) >> 31 ? 0xFFFFFFFF : 0x80000000)
 * ------------------------------------------------------------------------------------------- */

/* ---------------------------------------------------------------------------------------------
 * a1  Weight fake-quantization, multi-tensor (one launch pair for every layer).
 *     Replaces UniformQuantization.__uniform_quantize(mode='weight') + __scale + __inv_scale +
 *     __channel_bucket / __split_bucket — learners/uniform_quantization/utils.py:163-289.
 *
 *     Every tensor is described by one pf_uq_seg.  Bucket id of flat element i is (i % ncols):
 *       per-layer  (use_buckets=False): ncols = 1,              padded = numel
 *       'channel'  (reshape [-1,cout], reduce axis 0): ncols = cout, padded = numel
 *       'split'    (pad with copies of the LAST element to a multiple of bucket_size, reshape
 *                   [bucket_size,-1], reduce axis 0): ncols = padded/bucket_size; elements
 *                   i in [numel,padded) read src[numel-1]   (utils.py:247-274: strided buckets)
 *     qw = alpha*(rint((w-beta)/alpha*k)/k)+beta, alpha=(max-min)+1e-10f, beta=min,
 *     k=float(2^bits-1); round-half-even; every op individually rounded (no FMA contraction).
 * ------------------------------------------------------------------------------------------- */
typedef struct pf_uq_seg {
  const float* src;   /* device; 16-byte aligned                                  */
  float* dst;         /* device; 16-byte aligned; may equal src                   */
  int64_t numel;      /* < 2^31                                                    */
  int64_t padded;     /* >= numel; multiple of ncols                               */
  int32_t ncols;      /* number of buckets of this tensor                          */
  int32_t bucket0;    /* first slot of this tensor in mn_enc/mx_enc (multiple of 4)*/
  int32_t bits;       /* 1..32                                                     */
  int32_t reserved;
} pf_uq_seg;

/* One unit of CTA work.  kind 0: flat chunk [start, start+count) of seg (elementwise kernels and
 * per-layer min/max).  kind 1: column tile for bucketed min/max: columns [c0, c0+ncol_tile),
 * rows [start, start+count) of the [padded/ncols, ncols] view. */
typedef struct pf_work {
  int32_t seg;
  int32_t kind;
  int64_t start;
  int32_t count;
  int32_t c0;
  int32_t ncol_tile;
  int32_t reserved;
} pf_work;

/* Phase 1: per-bucket min/max into ordered-uint slots (caller pre-fills mn_enc with 0xFF bytes and
 * mx_enc with 0 — pf_fill_u32 does both).  work table = kind-0 chunks (per-layer) / kind-1 tiles. */
int pf_uq_weight_minmax(const pf_uq_seg* segs_dev, const pf_work* work_dev, int n_work,
                        uint32_t* mn_enc_dev, uint32_t* mx_enc_dev, void* stream);
/* Phase 1b: scales_dev[0..n) = alpha = (max-min)+1e-10f, [n..2n) = beta = min, [2n..3n) = RN(1/alpha)
 * (n = n_buckets, a multiple of 4).  The reciprocal feeds an exact (correctly rounded) division by
 * residual correction, so results stay bit-identical to true fp32 division. */
int pf_uq_weight_scales(const uint32_t* mn_enc_dev, const uint32_t* mx_enc_dev, int n_buckets,
                        float* scales_dev, void* stream);
/* Phase 2: quantize.  work table: kind-0 chunks.  (The second read of the weights is an L2 hit:
 * all weights of ResNet-50 are 94 MB < 126 MB L2.) */
int pf_uq_weight_quant(const pf_uq_seg* segs_dev, const pf_work* work_dev, int n_work,
                       const float* scales_dev, int n_buckets, void* stream);
/* a3  STE backward of the weight quantizer as a stand-alone op, in place on the gradient:
 *     g <- (((g*alpha)/k)*k)/alpha   (gradient_override_map Round->Identity, utils.py:185-186;
 *     min/max under stop_gradient, :224-225).  segs[i].src/dst point at the gradient. */
int pf_uq_weight_ste_bwd(const pf_uq_seg* segs_dev, const pf_work* work_dev, int n_work,
                         const float* scales_dev, int n_buckets, void* stream);

/* a2  Activation fake-quantization (per-TENSOR min/max, utils.py:51-79, 215-231).
 *     minmax: accumulates into minmax_enc_dev[0] (min) / [1] (max) (pre-filled 0xFFFFFFFF / 0).
 *     quant : y = Q(x) with the scalar range; src may equal dst. */
int pf_uq_act_minmax(const float* x_dev, int64_t n, uint32_t* minmax_enc_dev, void* stream);
int pf_uq_act_quant(const float* x_dev, float* y_dev, int64_t n, const uint32_t* minmax_enc_dev,
                    int bits, void* stream);
/* same, (also) writing y as split-bf16 planes for the tensor-core conv that consumes it (y_dev may be NULL) */
int pf_uq_act_quant_planes(const float* x_dev, float* y_dev, void* y_hi_dev, void* y_lo_dev, int64_t n,
                           const uint32_t* minmax_enc_dev, int bits, void* stream);

int pf_fill_u32(uint32_t* p_dev, int64_t n, uint32_t value, void* stream);
/* (min,max) ordered-uint pairs <- (0xFFFFFFFF, 0): one launch resets every activation range slot. */
int pf_minmax_reset(uint32_t* pairs_dev, int64_t n_pairs, void* stream);

/* ---------------------------------------------------------------------------------------------
 * a5  Magnitude-threshold mask build, multi-tensor.
 *     Replaces WeightSparseLearner.__build_masks — learners/weight_sparsification/learner.py:260-294:
 *        bkup = where(mask > 0.5, w, bkup); thr = percentile(|bkup|, 100*s) ('nearest': the
 *        element at index rank_desc of the DESCENDING sort); mask = float(|bkup| > thr);
 *        w = bkup*mask.
 *     The order statistic is found exactly by a 4-pass radix select on the IEEE bit pattern of
 *     |bkup| (no sort, no approximation) so masks are bit-exact.
 *     ranks_desc_dev[i] = clip(int32(rint((n-1)*(1-q/100))),0,n-1), computed on the host in
 *     float64 exactly as tf.contrib.distributions.percentile does.
 *     workspace_dev: n_seg * PF_WS_WORKSPACE_U32_PER_SEG uint32 (zeroed by the call).
 *     thr_out_dev (optional, n_seg floats) receives each tensor's threshold.
 * ------------------------------------------------------------------------------------------- */
typedef struct pf_ws_seg {
  float* w;
  float* bkup;
  float* mask;
  int64_t numel;
} pf_ws_seg;
#define PF_WS_WORKSPACE_U32_PER_SEG (256 + 8)

int pf_ws_mask_build(const pf_ws_seg* segs_dev, int n_seg, const pf_work* work_dev, int n_work,
                     const int64_t* ranks_desc_dev, uint32_t* workspace_dev, float* thr_out_dev,
                     void* stream);

/* Exact k-th order statistic of plain values (not |.|), multi-tensor, used by the codebook
 * quantile initialisation (learners/nonuniform_quantization/utils.py:349-366).  Query q reads
 * segs[qseg[q]].bkup (numel floats) and returns the element at descending index ranks_desc[q]. */
int pf_select_desc(const pf_ws_seg* segs_dev, const int32_t* qseg_dev, int n_query,
                   const pf_work* work_dev, int n_work, /* work[].seg indexes QUERIES */
                   const int64_t* ranks_desc_dev, uint32_t* workspace_dev, float* out_dev,
                   void* stream);

/* ---------------------------------------------------------------------------------------------
 * a6/a9  Fused optimizer steps over flat fp32 ranges.
 *   momentum: replaces __calc_grads_pruned (weight_sparsification/learner.py:314-332) +
 *     MomentumOptimizer.apply_gradients (:201,:212), with the Horovod average
 *     (utils/multi_gpu_wrapper.py:82-89) and the l2_loss gradient folded in:
 *        gt = g*grad_scale + wd*w ; gt *= mask (if mask) ; acc = acc*mom + gt ; w -= lr*acc
 *   adam: TF-1.x ApplyAdam (uniform_quantization/learner.py:244):
 *        gt as above (no mask); alpha = lr*sqrt(1-b2p)/(1-b1p);
 *        m += (gt-m)*(1-b1); v += (gt*gt-v)*(1-b2); w -= (m*alpha)/(sqrt(v)+eps)
 *   lr/b1p/b2p are read from device scalars (hp_dev) so the step is CUDA-graph replayable:
 *     momentum: hp_dev[0]=lr ; adam: hp_dev[0]=lr, [1]=beta1_power, [2]=beta2_power.
 * ------------------------------------------------------------------------------------------- */
int pf_momentum_step(float* w_dev, float* acc_dev, const float* g_dev, const float* mask_dev,
                     int64_t n, const float* hp_dev, float momentum, float wd, float grad_scale,
                     void* stream);
int pf_adam_step(float* w_dev, float* m_dev, float* v_dev, const float* g_dev, int64_t n,
                 const float* hp_dev, float beta1, float beta2, float eps, float wd,
                 float grad_scale, void* stream);

/* ---------------------------------------------------------------------------------------------
 * a7/a8  Losses.
 *   pf_softmax_ce_fwd_bwd replaces tf.losses.softmax_cross_entropy(onehot, logits)
 *     (nets/resnet_at_cifar10.py:104) and DistillationHelper.calc_loss
 *     (learners/distillation_helper.py:86-103) in one pass over the N x K logits:
 *        hard = mean_n CE(labels_n, s_n)
 *        dst  = w_dst * mean_n CE(softmax(t_n/T), s_n/T)        (teacher_dev may be NULL)
 *        dlogits = d(hard+dst)/ds ; correct_n = [argmax labels == argmax s]
 *     out_dev[0]=hard, [1]=dst, [2]=accuracy (top-1), [3]=top-5 accuracy.
 *     row_ws_dev: 4*N floats of scratch.  Deterministic (fixed-order final reduction).
 *   pf_l2_loss: out_dev[0] = scale * sum(v^2)/2 over a flat range (tf.nn.l2_loss summed by add_n,
 *     nets/resnet_at_cifar10.py:105-107).  partial_ws_dev: PF_L2_PARTIALS floats.
 * ------------------------------------------------------------------------------------------- */
int pf_softmax_ce_fwd_bwd(const float* logits_dev, const float* labels_dev,
                          const float* teacher_dev, int n, int k, float tempr, float w_dst,
                          float* dlogits_dev, float* out_dev, float* row_ws_dev, void* stream);
#define PF_L2_PARTIALS 1024
int pf_l2_loss(const float* v_dev, int64_t n, float scale, int accumulate, float* out_dev,
               float* partial_ws_dev, void* stream);

/* ---------------------------------------------------------------------------------------------
 * a11 Codebook (non-uniform) weight quantization, multi-tensor, per-layer range.
 *     Replaces NonUniformQuantization.__nonuni_quantize / __build_norm_quant_point —
 *     learners/nonuniform_quantization/utils.py:168-194, 284-307:
 *        xn=(w-beta)/alpha; idx=argmin_j|xn-c_j| (first index on ties);
 *        q=c[idx]*sign(xn+1e-6); out=alpha*q+beta.
 *     Uses pf_uq_seg (ncols must be 1; bits = log2(#centroids) <= 8) and the scales of
 *     pf_uq_weight_minmax + pf_uq_weight_scales.  clusters_dev: per seg 2^bits floats at offset seg*256.
 *     idx_out_dev (optional): uint8 centroid index per element, laid out like the weights
 *     (idx_base_dev[seg] = byte offset of the tensor), for the codebook gradient.
 * ------------------------------------------------------------------------------------------- */
int pf_nuq_weight_quant(const pf_uq_seg* segs_dev, const pf_work* work_dev, int n_work,
                        const float* scales_dev, int n_buckets,
                        const float* clusters_dev, uint8_t* idx_out_dev,
                        const int64_t* idx_base_dev, void* stream);
/* same, with the codebook of tensor `seg` at clusters_base_dev + cluster_off_dev[seg] (floats): codebooks that live
 * among the model's trainable variables (the reference's `clusters` variables, utils.py:297) */
int pf_nuq_weight_quant_ex(const pf_uq_seg* segs_dev, const pf_work* work_dev, int n_work,
                           const float* scales_dev, int n_buckets, const float* clusters_base_dev,
                           const int64_t* cluster_off_dev, uint8_t* idx_out_dev, const int64_t* idx_base_dev,
                           void* stream);
/* f4  Codebook gradient of the `cluster` / `both` optimisation modes (learners/nonuniform_quantization/
 *     learner.py:252-261): backward of tf.gather(c, min_index) under the Mul->Add / Sign->Identity override
 *     (utils.py:303-306) through the inverse scale alpha*q+beta (:433):
 *        dL/dc_j = alpha * sum_{i : idx_i = j} g_i ,   g = gradient w.r.t. the quantized tensor.
 *     gsegs[i].src = g of tensor i (numel floats; bits, bucket0 as in the forward's segs); work: kind-0 chunks, all
 *     chunks of a tensor contiguous, work_first_dev[seg .. seg+1) = its range (n_seg + 1 entries); idx/idx_base: what
 *     pf_nuq_weight_quant wrote; partial_ws_dev: n_work * 256 floats; result at grad_base_dev + cluster_off_dev[seg].
 *     Deterministic (fixed-order two-stage reduction). */
int pf_nuq_cluster_grad(const pf_uq_seg* gsegs_dev, int n_seg, const pf_work* work_dev, int n_work,
                        const int32_t* work_first_dev, const uint8_t* idx_dev, const int64_t* idx_base_dev,
                        const float* scales_dev, float* partial_ws_dev, float* grad_base_dev,
                        const int64_t* cluster_off_dev, void* stream);

/* a11b Bucketed codebooks (--nuql_use_buckets): NonUniformQuantization.__bucket_quantize /
 *     __build_bucket_norm_quant_point / __quantile_init(axis=0) — learners/nonuniform_quantization/utils.py:196-243,
 *     309-366.  One codebook per bucket (bucket of flat element i = i % ncols, the layout of pf_uq_seg with
 *     split / channel buckets) and the per-bucket scales of pf_uq_weight_minmax + pf_uq_weight_scales.  The
 *     codebooks of tensor `seg` are the [2^bits', ncols] row-major `clusters` variable at
 *     clusters_base_dev + cluster_off_dev[seg] (bits' >= bits): centroid j of bucket b at + j*ncols + b.
 *
 *     Quantize: work = kind-1 column tiles (rows [start, start+count) x columns [c0, c0+ncol_tile) of the
 *     [padded/ncols, ncols] view) with (2^bits + 3) * ncol_tile <= PF_NUQ_BUCKET_TILE_FLOATS + 3 * ncol_tile and
 *     ncol_tile <= PF_NUQ_BUCKET_MAX_TILE.  Only elements with flat index < numel are written; idx_out as in
 *     pf_nuq_weight_quant. */
#define PF_NUQ_BUCKET_TILE_FLOATS 8192
#define PF_NUQ_BUCKET_MAX_TILE 1024
#define PF_NUQ_BUCKET_MAX_ROWS 16384
#define PF_NUQ_BUCKET_GRAD_TILE 32
int pf_nuq_bucket_weight_quant(const pf_uq_seg* segs_dev, const pf_work* work_dev, int n_work,
                               const float* scales_dev, int n_buckets, const float* clusters_base_dev,
                               const int64_t* cluster_off_dev, uint8_t* idx_out_dev, const int64_t* idx_base_dev,
                               void* stream);
/* Quantile init, one CTA per bucket slot (n_buckets = the scales' slot count): centroid j of bucket b =
 *     x_n at descending rank ranks_dev[seg*256 + j] of the bucket's padded/ncols rows (padding rows = copies of the
 *     last element, counted as the reference counts them), x_n = (w-beta)/alpha in fp32.  Writes rows 0..2^bits-1 of
 *     each codebook.  max_rows = the tallest bucket, at most PF_NUQ_BUCKET_MAX_ROWS (sorted in shared memory). */
int pf_nuq_bucket_quantile_init(const pf_uq_seg* segs_dev, int n_seg, const float* scales_dev, int n_buckets,
                                const int32_t* ranks_dev, int max_rows, float* clusters_base_dev,
                                const int64_t* cluster_off_dev, void* stream);
/* Codebook gradient, dL/dc[j,b] = alpha_b * sum_{i < numel, i % ncols = b, idx_i = j} g_i.  work: kind-1 tiles of at
 *     most PF_NUQ_BUCKET_GRAD_TILE columns x a row range; tiles_dev[t]: seg, c0, ncol_tile of column tile t and, in
 *     start/count, the contiguous range of its work items; partial_ws_dev: n_work * kmax * PF_NUQ_BUCKET_GRAD_TILE
 *     floats (kmax >= every 2^bits).  Deterministic (fixed-order two-stage reduction); writes only rows 0..2^bits-1
 *     of the codebooks in grad_base_dev (layout of clusters_base_dev). */
int pf_nuq_bucket_cluster_grad(const pf_uq_seg* gsegs_dev, const pf_work* work_dev, int n_work,
                               const pf_work* tiles_dev, int n_tiles, int kmax, const uint8_t* idx_dev,
                               const int64_t* idx_base_dev, const float* scales_dev, float* partial_ws_dev,
                               float* grad_base_dev, const int64_t* cluster_off_dev, void* stream);

/* ---------------------------------------------------------------------------------------------
 * a4  Convolution / dense layers, exact-fp32 CUDA-core path (pf_conv.cu).
 *     Replaces tf.nn.conv2d / tf.matmul re-created on the quantized weight
 *     (learners/uniform_quantization/utils.py:88-113) and their autodiff (learner.py:247).
 *     x: NHWC [n,h,w,c]; w: HWIO [r,s,c,k]; y: NHWC [n,p,q,k]; pad_t/pad_l = leading padding
 *     (TF 'SAME': pad_total//2; fixed_padding: (k-1)//2 — utils/external/resnet_model.py:71-103).
 *     A dense layer is the h=w=r=s=1 case.
 * ------------------------------------------------------------------------------------------- */
typedef struct pf_conv_desc {
  int32_t n, h, w, c;      /* input  */
  int32_t k, r, s;         /* filters, kernel height/width */
  int32_t p, q;            /* output height/width */
  int32_t stride_h, stride_w, pad_t, pad_l;
} pf_conv_desc;            /* HOST struct, passed by pointer */
#define PF_CONV_WGRAD_MAX_SPLITS 64
#define PF_BN_MAX_SPLITS 1024

/* cols[m][k] (m = output pixel, k = (r*S+s)*C + c, zero-padded to kpad columns): explicit im2col for
 * first layers whose Cin (3) the tensor-core path cannot take; the conv then runs as a 1x1 conv over
 * kpad channels. */
int pf_im2col(const pf_conv_desc* d, const float* x_dev, int kpad, float* cols_dev, void* stream);
/* Space-to-depth form of a stride-2 first layer: x' [n, hp, wp, cpad] (split-bf16 planes) with
 * x'[.., y', x', (dy*2+dx)*c + cc] = x[.., 2y'+dy-pad_t, 2x'+dx-pad_l, cc]; the RxS stride-2 conv equals a stride-1
 * ceil(R/2) x ceil(S/2) conv over x' whose kernel rows are re-arranged with pf_gather_rows (idx < 0: zero row). */
int pf_s2d_planes(const float* x_dev, int n, int h, int w, int c, int pad_t, int pad_l, int hp, int wp, int cpad,
                  void* hi_dev, void* lo_dev, void* stream);
int pf_gather_rows(const float* src_dev, const int32_t* idx_dev, int n_rows, int row_len, float* dst_dev, void* stream);
/* same, written directly as split-bf16 operand planes [N*P*Q, kpad] (kpad % 8 == 0) */
int pf_im2col_planes(const pf_conv_desc* d, const float* x_dev, int kpad, void* cols_hi_dev, void* cols_lo_dev,
                     void* stream);
/* y = conv(x, w) (+ bias[k]) (relu if relu != 0) */
int pf_conv2d_fwd(const pf_conv_desc* d, const float* x_dev, const float* w_dev, const float* bias_dev,
                  int relu, float* y_dev, void* stream);
/* dx (+)= conv_transpose(dy, w).  wt_ws_dev: r*s*c*k floats of scratch (per-tap transposed weight). */
int pf_conv2d_dgrad(const pf_conv_desc* d, const float* dy_dev, const float* w_dev, float* wt_ws_dev,
                    int accumulate, float* dx_dev, void* stream);
/* dw = x (*) dy, split-K with a fixed-order reduction (deterministic).
 * ws_dev: pf_conv2d_wgrad_workspace_bytes(d) bytes. */
int64_t pf_conv2d_wgrad_workspace_bytes(const pf_conv_desc* d);
int pf_conv2d_wgrad(const pf_conv_desc* d, const float* x_dev, const float* dy_dev, float* ws_dev,
                    float* dw_dev, void* stream);

/* ---------------------------------------------------------------------------------------------
 * a4  Convolution forward / dgrad on the tcgen05 tensor cores (pf_conv_tc.cu), same semantics as
 *     pf_conv2d_fwd / pf_conv2d_dgrad.  fp32 operands are split x = hi + lo (bf16 each) and each
 *     k-slice issues hi*hi + hi*lo + lo*hi into one fp32 TMEM accumulator (error ~2^-17 relative).
 *     Requires Cin % 16 == 0 and Cout % 16 == 0 (pf_conv2d_tc_supported).
 *     Weights are pre-split and laid out K-major once per step by pf_conv2d_tc_prep_weight into
 *     caller-owned bf16 buffers of pf_conv2d_tc_weight_elems(d, dgrad) elements each, which the caller
 *     zero-fills ONCE at allocation (padding columns are never written).
 * ------------------------------------------------------------------------------------------- */
int pf_conv2d_tc_supported(const pf_conv_desc* d);
int64_t pf_conv2d_tc_weight_elems(const pf_conv_desc* d, int dgrad);
int pf_conv2d_tc_prep_weight(const pf_conv_desc* d, const float* w_dev, void* fwd_hi_dev, void* fwd_lo_dev,
                             void* dgrad_hi_dev, void* dgrad_lo_dev, void* stream);
/* y = conv(x, w) (+ bias) (relu) (+ residual_dev: the fused residual add of resnet_model.py:199,314;
 * NULL = none) */
int pf_conv2d_tc_fwd(const pf_conv_desc* d, const float* x_dev, const void* w_hi_dev, const void* w_lo_dev,
                     const float* bias_dev, int relu, const float* residual_dev, float* y_dev, void* stream);
int pf_conv2d_tc_dgrad(const pf_conv_desc* d, const float* dy_dev, const void* wd_hi_dev, const void* wd_lo_dev,
                       int accumulate, float* dx_dev, void* stream);
/* multi-tensor weight preparation: every conv kernel of a network in ONE launch.  segs: one entry per kernel
 * (kpad = pf_conv2d_tc_weight_elems / rows; dgrad pointers may be NULL), work: one item per 32 x 64 tile of the
 * [R*S*Cin, Cout] matrix (start = first row, c0 = first column). */
typedef struct pf_tc_prep_seg {
  const float* w;          /* HWIO fp32 */
  void* fwd_hi;
  void* fwd_lo;
  void* dgrad_hi;
  void* dgrad_lo;
  int32_t rs, c, k;        /* R*S, Cin, Cout */
  int32_t kpad_f, kpad_d;  /* row pitches of the fwd / dgrad copies (multiples of 64) */
  int32_t q_bits;          /* 0: w holds the values to split.  1..8: w holds the UNQUANTIZED kernel and the copies are
                            * derived with the weight quantizer's own op chain (a1): fwd_hi <- bf16(level - 2^(bits-1))
                            * (integer levels, fwd_lo untouched), dgrad_hi / dgrad_lo <- split of the quantized value */
  const float* q_alpha;    /* bucket scales of pf_uq_weight_scales at this tensor's first bucket: alpha, */
  const float* q_beta;     /*   beta, */
  const float* q_ralpha;   /*   RN(1 / alpha) */
  int32_t q_ncols;         /* 1 (per layer) or k (per output channel) */
  int32_t reserved;
} pf_tc_prep_seg;
int pf_conv2d_tc_prep_weights_multi(const pf_tc_prep_seg* segs_dev, const pf_work* work_dev, int n_work, void* stream);
/* dw = x (*) dy on the tensor cores (MN-major operands, split-K with a fixed-order reduction).
 * Requires Cin % 16 == 0 and Cout % 64 == 0; ws_dev: pf_conv2d_tc_wgrad_workspace_bytes(d) bytes. */
#define PF_CONV_TC_WGRAD_MAX_SPLITS 148
int pf_conv2d_tc_wgrad_supported(const pf_conv_desc* d);
int64_t pf_conv2d_tc_wgrad_workspace_bytes(const pf_conv_desc* d);
int pf_conv2d_tc_wgrad(const pf_conv_desc* d, const float* x_dev, const float* dy_dev, float* ws_dev,
                       float* dw_dev, void* stream);
/* fp32 -> split-bf16 planes: hi = bf16(x), lo = bf16(x - hi) (n % 8 == 0, 16-byte aligned); the operand format of
 * the tensor-core kernels.  pf_conv2d_tc_wgrad splits x and dy into its workspace and then runs the same
 * persistent kernel as pf_conv2d_tc_wgrad_planes, which takes operands that are already split. */
int pf_split_bf16(const float* src_dev, void* hi_dev, void* lo_dev, int64_t n, void* stream);
int64_t pf_conv2d_tc_wgrad_planes_workspace_bytes(const pf_conv_desc* d);   /* split-K partials only */
/* the same fwd / dgrad kernels with the activation operand already split (written by pf_bn_apply_planes,
 * pf_uq_act_quant_planes, pf_bn_bwd_planes or pf_split_bf16): producers are pure cp.async copies */
int pf_conv2d_tc_fwd_planes(const pf_conv_desc* d, const void* x_hi_dev, const void* x_lo_dev, const void* w_hi_dev,
                            const void* w_lo_dev, const float* bias_dev, int relu, const float* residual_dev,
                            float* y_dev, void* stream);
int pf_conv2d_tc_dgrad_planes(const pf_conv_desc* d, const void* dy_hi_dev, const void* dy_lo_dev, const void* wd_hi_dev,
                              const void* wd_lo_dev, int accumulate, float* dx_dev, void* stream);
/* dw_dev == NULL: leave the split-K partials [splits][R*S*Cin][Cout] in ws_dev (pf_conv2d_tc_wgrad_splits(d) of
 * them) for ONE deferred pf_conv2d_tc_wgrad_reduce_multi over every layer of the step */
typedef struct pf_tc_reduce_seg {
  const float* partial;    /* [splits][n] */
  float* out;              /* [n] */
  int64_t n;               /* multiple of 4 */
  int32_t splits;
  int32_t reserved;
} pf_tc_reduce_seg;
int pf_conv2d_tc_wgrad_splits(const pf_conv_desc* d);
int pf_conv2d_tc_wgrad_reduce_multi(const pf_tc_reduce_seg* segs_dev, const pf_work* work_dev, int n_work, void* stream);
int pf_conv2d_tc_wgrad_planes(const pf_conv_desc* d, const void* x_hi_dev, const void* x_lo_dev, const void* dy_hi_dev,
                              const void* dy_lo_dev, float* ws_dev, float* dw_dev, void* stream);
/* ---- TMA-fed kernels with EXACT quantizer-level operands (pf_conv_tma.cu; SURVEY §7 hard part 1b) ----
 * When channel counts are multiples of 64 the same entry points above feed the tensor cores with TMA
 * (cp.async.bulk.tensor: im2col-mode tensor maps for the NHWC operand, tiled maps for the weight / gradient matrices;
 * PF_TC_FEED=lsu forces the cp.async kernels).  The *_ex entry points additionally accept operands of <= 8-bit
 * fake-quantized tensors as their INTEGER LEVELS, which bf16 represents exactly, so one MMA per k-slice replaces
 * three (two where the other operand is a split-bf16 gradient):
 *   activation (reference: learners/uniform_quantization/utils.py:51-79, 175-199):  qa = scale * level,
 *     plane0 = levels (plane1 unused) when the tensor's minimum is 0, otherwise plane0/plane1 = hi/lo of qa and
 *     scale = 1 — the producer (pf_bn_apply_quant_levels) decides on the device and records it in `hdr`;
 *     csum[pixel][nseg] = sums of the stored plane values over channel segments of min(C,128) (for the rank-1
 *     correction that the weight offset needs: sum_k qa[m,k] over the filter window);
 *   weights (utils.py:81-113, 224-245):  qw = (alpha_c / k) (level - centre) + (beta_c + centre alpha_c / k),
 *     plane0 = bf16(level - centre), centre = 2^(bits-1), k = 2^bits - 1; alpha / beta = the quantizer's bucket
 *     scales (per layer or per output channel).  plane1 != NULL, alpha == NULL: plain split-bf16 weights. */
typedef struct pf_tc_act_hdr {
  float scale;             /* value of one level (1.0 when the planes hold hi / lo) */
  int32_t nplanes;         /* 1: plane0 = integer levels; 2: plane0 / plane1 = hi / lo */
} pf_tc_act_hdr;
typedef struct pf_tc_act {
  const void* plane0;      /* bf16, layout of the fp32 tensor */
  const void* plane1;      /* bf16 or NULL (then hdr must say 1 plane, or hdr == NULL and the tensor is bf16-exact) */
  const pf_tc_act_hdr* hdr;/* device, or NULL: nplanes = (plane1 ? 2 : 1), scale = 1 */
  const float* csum;       /* device [pixels][nseg] or NULL (only needed with weight levels) */
  int32_t nseg;
  int32_t reserved;
} pf_tc_act;
typedef struct pf_tc_wt {
  const void* plane0;      /* bf16 K-major [rows][kpad] as written by pf_conv2d_tc_prep_weight* */
  const void* plane1;      /* lo plane, or NULL with levels */
  const float* alpha;      /* device bucket scales (levels) or NULL */
  const float* beta;
  int32_t per_channel;     /* 1: one bucket per output channel; 0: one per layer */
  int32_t bits;
} pf_tc_wt;
int pf_conv2d_tc_tma_supported(const pf_conv_desc* d, int pass /* 0 fwd, 1 dgrad, 2 wgrad */);
/* producer of a pf_tc_act: Q(act(bn(x))) with a known range (as pf_bn_apply_quant), written as levels / planes +
 * header + channel sums (csum_dev: m * ceil(c / 128) floats).  C must be a power of two >= 16.  y_dev (fp32 copy) may
 * be NULL.  Reference ops: utils/external/resnet_model.py:55-62 + learners/uniform_quantization/utils.py:51-79. */
int pf_bn_apply_quant_levels(const float* x_dev, int64_t m, int c, const float* mean_dev, const float* rstd_dev,
                             const float* gamma_dev, const float* beta_dev, int act, const uint32_t* range_enc_dev,
                             int bits, float* y_dev, void* plane0_dev, void* plane1_dev, pf_tc_act_hdr* hdr_dev,
                             float* csum_dev, void* stream);
/* operand feed of the tensor-core kernels: 1 = TMA where eligible (default), 0 = cp.async everywhere, -1 = back to the
 * PF_TC_FEED environment default.  Process-wide; used by the tests to run both kernels on the same inputs. */
int pf_conv2d_tc_set_feed(int mode);
int pf_conv2d_tc_fwd_ex(const pf_conv_desc* d, const pf_tc_act* x, const pf_tc_wt* w, const float* bias_dev, int relu,
                        const float* residual_dev, float* y_dev, void* stream);
int pf_conv2d_tc_dgrad_ex(const pf_conv_desc* d, const pf_tc_act* dy, const pf_tc_wt* wd, int accumulate, float* dx_dev,
                          void* stream);
int pf_conv2d_tc_wgrad_ex(const pf_conv_desc* d, const pf_tc_act* x, const pf_tc_act* dy, float* ws_dev, float* dw_dev,
                          void* stream);
/* hardware probe used by tests/test_tc_gpu.py to pin the descriptor conventions (not a product op) */
int pf_tc_probe(const void* a_dev, const void* b_dev, float* d_dev, int n, int k, int mode, uint32_t lbo_a,
                uint32_t sbo_a, uint32_t lbo_b, uint32_t sbo_b, uint32_t kstep_a, uint32_t kstep_b, void* stream);

/* ---------------------------------------------------------------------------------------------
 * a4  Depthwise convolution, depth multiplier 1 (pf_dwconv.cu): slim.separable_conv2d's depthwise half
 *     (utils/external/mobilenet_v1.py:273-280; TF op DepthwiseConv2dNative).  x NHWC, w [r,s,c,1],
 *     descriptor with k == c, c % 4 == 0, r*s <= 9.  HBM-bound.  wgrad: ws_dev of
 *     pf_dwconv_wgrad_workspace_bytes(d) bytes; deterministic.
 * ------------------------------------------------------------------------------------------- */
#define PF_DWCONV_MAX_SPLITS 1024
int pf_dwconv_fwd(const pf_conv_desc* d, const float* x_dev, const float* w_dev, float* y_dev, void* stream);
int pf_dwconv_dgrad(const pf_conv_desc* d, const float* dy_dev, const float* w_dev, int accumulate, float* dx_dev,
                    void* stream);
int64_t pf_dwconv_wgrad_workspace_bytes(const pf_conv_desc* d);
int pf_dwconv_wgrad(const pf_conv_desc* d, const float* x_dev, const float* dy_dev, float* ws_dev, float* dw_dev,
                    void* stream);

/* ---------------------------------------------------------------------------------------------
 * a13 The HBM-bound layers between the convolutions (pf_nn.cu); tensors viewed as [m, c], c % 4 == 0.
 *     tf.layers.batch_normalization(momentum, eps, fused) — utils/external/resnet_model.py:55-62:
 *       stats : batch mean / biased variance / rstd (+ moving-stat update, unbiased moving variance);
 *               ws_dev: 3*c*PF_BN_MAX_SPLITS floats.
 *       apply : y = act(((x-mean)*rstd)*gamma+beta), act 0 none / 1 relu / 2 relu6; when
 *               minmax_enc_dev != NULL also accumulates the per-tensor min/max of y for the
 *               activation quantizer (utils.py:51-79) — the reference's two extra reduction passes.
 *       bwd   : dgamma, dbeta, dx (+)= through act and training-mode BN; ws_dev as for stats.
 * ------------------------------------------------------------------------------------------- */
int pf_bn_train_stats(const float* x_dev, int64_t m, int c, float eps, float momentum, float* mean_dev,
                      float* var_dev, float* rstd_dev, float* moving_mean_dev, float* moving_var_dev,
                      float* ws_dev, void* stream);
/* stats + the per-tensor range of y = act(bn(x)) for the activation quantizer, evaluated from the per-channel
 * extremes of x (every step of bn/act is monotone in x, so the result is bit-identical to a min/max pass over
 * y); accumulates into minmax_enc_dev[0..1] (ordered-uint).  ws_dev: 5 * C * PF_BN_MAX_SPLITS floats. */
int pf_bn_train_stats_range(const float* x_dev, int64_t m, int c, float eps, float momentum, float* mean_dev,
                            float* var_dev, float* rstd_dev, float* moving_mean_dev, float* moving_var_dev,
                            const float* gamma_dev, const float* beta_dev, int act, uint32_t* minmax_enc_dev,
                            float* ws_dev, void* stream);
int pf_bn_eval_prepare(const float* moving_var_dev, int c, float eps, float* rstd_dev, void* stream);
/* inference-mode BN in one launch: rstd = rsqrt(moving_var + eps) is formed in the kernel (same roundings as
 * pf_bn_eval_prepare + pf_bn_apply); fp32 and/or split-bf16 plane output */
int pf_bn_apply_eval(const float* x_dev, int64_t m, int c, const float* moving_mean_dev, const float* moving_var_dev,
                     float eps, const float* gamma_dev, const float* beta_dev, int act, float* y_dev, void* y_hi_dev,
                     void* y_lo_dev, uint32_t* minmax_enc_dev, void* stream);
/* y = Q(act(bn(x))) in one pass with a known range (pf_bn_train_stats_range): fp32 and/or split-bf16 planes */
int pf_bn_apply_quant(const float* x_dev, int64_t m, int c, const float* mean_dev, const float* rstd_dev,
                      const float* gamma_dev, const float* beta_dev, int act, const uint32_t* range_enc_dev, int bits,
                      float* y_dev, void* y_hi_dev, void* y_lo_dev, void* stream);
int pf_bn_apply(const float* x_dev, int64_t m, int c, const float* mean_dev, const float* rstd_dev,
                const float* gamma_dev, const float* beta_dev, int act, float* y_dev,
                uint32_t* minmax_enc_dev, void* stream);
int pf_bn_bwd(const float* dy_dev, const float* x_dev, int64_t m, int c, const float* mean_dev,
              const float* rstd_dev, const float* gamma_dev, const float* beta_dev, int act,
              float* dgamma_dev, float* dbeta_dev, float* dx_dev, int accumulate, float* ws_dev,
              void* stream);
/* variants that (also) write the result as split-bf16 planes — the operand format of the tensor-core convs that
 * consume it (y: next conv's fwd + wgrad; dx: the producing conv's dgrad + wgrad).  The fp32 output pointer may
 * be NULL when every consumer takes planes; `accumulate` needs the fp32 dx. */
int pf_bn_apply_planes(const float* x_dev, int64_t m, int c, const float* mean_dev, const float* rstd_dev,
                       const float* gamma_dev, const float* beta_dev, int act, float* y_dev, void* y_hi_dev,
                       void* y_lo_dev, uint32_t* minmax_enc_dev, void* stream);
int pf_bn_bwd_planes(const float* dy_dev, const float* x_dev, int64_t m, int c, const float* mean_dev,
                     const float* rstd_dev, const float* gamma_dev, const float* beta_dev, int act,
                     float* dgamma_dev, float* dbeta_dev, float* dx_dev, int accumulate, void* dx_hi_dev,
                     void* dx_lo_dev, float* ws_dev, void* stream);
/* out (+)= a (+ b): residual add (resnet_model.py:199,314) / gradient fan-out; b_dev may be NULL */
int pf_add(const float* a_dev, const float* b_dev, int64_t n, int accumulate, float* out_dev, void* stream);
/* dst[i][j] = sum_b src[b*m+i][b*n+j] (src is (g*m) x (g*n) row-major): folds the diagonal blocks of a weight gradient that
 * the tensor cores computed from g pixels per GEMM row (convs with fewer than 64 output channels) */
int pf_fold_diag_blocks(const float* src_dev, int g, int m, int n, float* dst_dev, void* stream);
/* dx (+)= dy * [y > 0] (and [y < 6] for act == 2) */
int pf_relu_bwd(const float* dy_dev, const float* y_dev, int64_t n, int act, int accumulate, float* dx_dev,
                void* stream);
/* out[c] = sum_m a[m][c] (bias gradient) */
int pf_colsum(const float* a_dev, int64_t m, int c, float* out_dev, void* stream);
/* max pooling (kernel r x s, strides, leading pads from the descriptor; k unused; c % 4 == 0).  The
 * forward records the window position of the FIRST maximum in row-major order (uint8 per output
 * element; argmax_dev may be NULL for inference) and the backward routes each gradient there, like
 * TF's MaxPoolGrad.  Gather form, deterministic. */
int pf_maxpool_fwd(const pf_conv_desc* d, const float* x_dev, float* y_dev, uint8_t* argmax_dev, void* stream);
int pf_maxpool_bwd(const pf_conv_desc* d, const float* dy_dev, const uint8_t* argmax_dev, int accumulate,
                   float* dx_dev, void* stream);
/* ILSVRC-12 preprocessing of a mini-batch of decoded uint8 RGB crops in one launch — what
 * utils/external/imagenet_preprocessing.py:225-260 does after decoding: TF1 bilinear resize (align_corners=False, no
 * half-pixel centres) of the [h, w, 3] crop at crops_dev + offset to [rh, rw], optional left-right flip of the SOURCE
 * (training flips before resizing), the [out_h, out_w] window at (top, left) of the resized image (evaluation:
 * central crop of the 256-short-side resize; training: rh = out_h, rw = out_w, top = left = 0), minus the channel
 * means.  dst_dev: fp32 [n, out_h, out_w, 3].  Bit-identical to the host restatement in
 * pocketflow_b200/datasets/ilsvrc12_dataset.py (every operation individually rounded). */
typedef struct pf_img_desc {
  int64_t offset;        /* byte offset of this crop in crops_dev */
  int32_t h, w;          /* crop size */
  int32_t rh, rw;        /* size it is resized to */
  int32_t top, left;     /* window origin inside the resized image */
  int32_t flip;          /* != 0: mirror the crop left-right before resizing */
  int32_t reserved;
} pf_img_desc;
int pf_preprocess_images(const uint8_t* crops_dev, const pf_img_desc* desc_dev, int n, int out_h, int out_w,
                         float mean_r, float mean_g, float mean_b, float* dst_dev, void* stream);
/* tf.reduce_mean over H,W (resnet_model.py:547-548) */
int pf_global_avgpool_fwd(const float* x_dev, int n, int hw, int c, float* y_dev, void* stream);
int pf_global_avgpool_bwd(const float* dy_dev, int n, int hw, int c, int accumulate, float* dx_dev, void* stream);
/* row softmax and its backward (nets/lenet_at_cifar10.py:66) */
int pf_softmax_fwd(const float* x_dev, int n, int k, float* y_dev, void* stream);
int pf_softmax_bwd(const float* dy_dev, const float* y_dev, int n, int k, float* dx_dev, void* stream);

/* ---------------------------------------------------------------------------------------------
 * f4  Layer-wise channel selection of the channel-pruning learner (pf_cpg.cu).
 *     Replaces, per proximal-gradient iteration of ChannelPrunedGpuLearner.__choose_channels
 *     (learners/channel_pruning_gpu/learner.py:445-518), the TF ops of __build_extra_losses (:339-354) and
 *     __build_layer_ops (:356-402); kernels W are [R,S,Cin,Cout] row-major, rs = R*S:
 *   pf_cpg_diff_l2     diff = a - b ; loss[0] = sum(diff^2)/2    (tf.nn.l2_loss of the two conv outputs, :352;
 *                      with a = pruned, b = full, diff is also d loss / d a).  partial_ws: PF_L2_PARTIALS floats.
 *   pf_cpg_group_norms norms[c] = sqrt(sum_{rs,k} (w - lr*g)^2)  (:378-379; g NULL: the norm of w itself, :256)
 *   pf_cpg_prox_apply  w = (w - lr*g) * max(1 - thr[0] / norms[c], 0)   (:378-382; thr = the percentile of norms)
 *   pf_cpg_channel_mask mask[rs,c,k] = norms[c] > 0               (:256-259)
 *   pf_mul             out = a * b                                 (masked gradient g * mask, :438)
 * ------------------------------------------------------------------------------------------- */
int pf_cpg_diff_l2(const float* a_dev, const float* b_dev, int64_t n, float* diff_dev, float* loss_dev,
                   float* partial_ws_dev, void* stream);
int pf_cpg_group_norms(const float* w_dev, const float* g_dev, float lr, int rs, int cin, int cout,
                       float* norms_dev, void* stream);
int pf_cpg_prox_apply(float* w_dev, const float* g_dev, float lr, const float* norms_dev, const float* thr_dev,
                      int rs, int cin, int cout, void* stream);
int pf_cpg_channel_mask(const float* norms_dev, int rs, int cin, int cout, float* mask_dev, void* stream);
int pf_mul(const float* a_dev, const float* b_dev, int64_t n, float* out_dev, void* stream);

/* ---------------------------------------------------------------------------------------------
 * a10 The collective of the data-parallel step (pf_comm.cu).  Replaces mgw.DistributedOptimizer's per-variable
 *     Horovod all-reduces and mgw.broadcast_global_variables (utils/multi_gpu_wrapper.py:82-98; call sites
 *     learners/uniform_quantization/learner.py:245-247, :271): ONE in-place ncclAllReduce (sum, fp32) over the flat
 *     gradient buffer — or over contiguous buckets of it as the backward pass completes them — enqueued on the
 *     caller's stream (CUDA-graph capturable); the division by the worker count is the optimizers' grad_scale.
 *     NCCL (libnccl.so.2, or the path in PF_NCCL_LIB) is bound at run time, not linked.
 *       pf_comm_unique_id  rank 0: 128 bytes to distribute to every rank (any host-side channel)
 *       pf_comm_init       collective over all ranks, on the calling thread's current device; *comm_out = handle
 *       pf_allreduce_flat / pf_broadcast_flat   asynchronous on `stream`
 * ------------------------------------------------------------------------------------------- */
int pf_comm_nccl_version(int* version_out);
int pf_comm_unique_id(void* id128_out);
int pf_comm_init(const void* id128, int n_ranks, int rank, void** comm_out);
int pf_comm_destroy(void* comm);
int pf_allreduce_flat(void* comm, float* buf_dev, int64_t n, void* stream);
int pf_broadcast_flat(void* comm, float* buf_dev, int64_t n, int root, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PF_B200_H_ */
