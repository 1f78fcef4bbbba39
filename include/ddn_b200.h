/* ddn_b200.h -- C ABI of the B200-native dense-descriptor training path.
 *
 * One shared library (libddn_b200.so, sm_100a only) exports everything below with C linkage:
 * plain pointers and sizes, no torch / C++ types.  All pointers are DEVICE pointers unless the
 * name ends in _host; `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 * Every function returns 0 on success, a negative DDN_E* code on a contract violation and a
 * positive cudaError_t when the CUDA runtime reports one; ddn_last_error() gives the text.
 * Nothing here allocates device memory: the caller owns every buffer (workspace sizes are
 * queried first) -- the host side above this boundary uses torch only as the allocator.
 *
 * The reference has no native code on this path (SURVEY.md 2c); each entry point replaces the
 * PyTorch-1.1 -> ATen -> cuDNN call sequence of the reference Python cited next to it
 * (paths relative to the reference root; PSD = external/pytorch-segmentation-detection).
 */
#ifndef DDN_B200_H_
#define DDN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DDN_ABI_VERSION 3

enum {
  DDN_OK = 0,
  DDN_EINVAL = -1,     /* bad shape / flag / null pointer            */
  DDN_EWORKSPACE = -2, /* workspace too small                         */
  DDN_EUNSUPPORTED = -3
};

/* Arithmetic used by the convolution contractions. */
enum {
  DDN_PRECISION_FP32_SIMT = 0, /* fp32 FFMA on CUDA cores (bit-for-bit class of the fp32 oracle)        */
  DDN_PRECISION_BF16X3 = 1,    /* tcgen05, operands split hi+lo bf16, 3 MMAs, fp32 accumulate in TMEM   */
  DDN_PRECISION_BF16 = 2       /* tcgen05, single bf16 pass ("fast mode"; fails the 1e-3 descriptor gate) */
};

int ddn_abi_version(void);
const char* ddn_last_error(void);

/* ------------------------------------------------------------------------------------------
 * Parameter layout of Resnet34_8s(num_classes=D)
 *   PSD/pytorch_segmentation_detection/models/resnet_dilated.py:283-322
 *   PSD/vision/torchvision/models/resnet.py:112-229 (names, shapes, order of named_parameters())
 * Learnable parameters live in ONE flat fp32 array, BatchNorm running statistics in a second one;
 * entry i of the tables gives the reference state-dict key (without the leading "resnet34_8s."),
 * its shape and its element offset in the flat array.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  char name[64];
  int32_t ndim;
  int32_t shape[4];
  int64_t offset; /* elements */
  int64_t numel;
} ddn_tensor_entry;

/* Fills up to `cap` entries, returns the number of learnable tensors (110). */
int ddn_resnet34_8s_param_table(int D, ddn_tensor_entry* out, int cap);
/* Running mean / running var entries (72 = 36 BN x 2), same convention. */
int ddn_resnet34_8s_buffer_table(ddn_tensor_entry* out, int cap);
int64_t ddn_resnet34_8s_param_count(int D);
int64_t ddn_resnet34_8s_buffer_count(void);

/* ------------------------------------------------------------------------------------------
 * Backbone forward / backward.
 *   forward  replaces Resnet34_8s.forward            (resnet_dilated.py:310-322)
 *                     ResNet.forward / BasicBlock    (resnet.py:231-265, :53-69)
 *            as called by DenseCorrespondenceNetwork.forward
 *                     (dense_correspondence/network/dense_correspondence_network.py:239-263)
 *   backward replaces the autograd backward of the same (dense_correspondence/training/training.py:345)
 *
 * x  [B,3,H,W] fp32 NCHW (already mean/std normalised), y [B,D,H,W] fp32 NCHW contiguous.
 * H, W multiples of 8 (the trunk runs at H/8 x W/8).  1 <= D <= 32.
 * mode DDN_MODE_TRAIN: BatchNorm uses the statistics of THIS call's images (biased variance) and updates
 *   running_mean/var in `buffers` with `momentum` and the unbiased variance, exactly like
 *   nn.BatchNorm2d in train(); the activations needed by backward are kept in `workspace`.
 * mode DDN_MODE_INFER: BatchNorm uses `buffers` (folded into the conv epilogues); nothing is kept.
 * mode DDN_MODE_EVAL_SAVE: BatchNorm uses `buffers` (frozen statistics) and the activations are kept, so that
 *   ddn_resnet34_8s_backward can differentiate an eval()-mode network like autograd does for the reference.
 * bn_groups G (1 or 2): the batch is G consecutive groups of B/G images, each normalised by its OWN batch
 *   statistics -- G = 2 runs the reference's two forward calls of a step (image A batch, image B batch:
 *   dense_correspondence/training/training.py:329-333) as one launch sequence; running statistics are updated
 *   group 0 first, then group 1, as the two calls would.
 * The same `workspace` (untouched in between) must be handed to ddn_resnet34_8s_backward (same mode / bn_groups),
 * which OVERWRITES grads[0 .. param_count) with dL/dparams for the cotangent dy [B,D,H,W].
 * on_bucket (may be NULL) is called on the HOST, in order, each time a contiguous range of `grads` is final --
 *   i.e. right after the last kernel writing grads[offset, offset+numel) has been enqueued on `stream` -- so that a
 *   data-parallel caller can start the all-reduce of that range while the rest of the backward still runs
 *   (4 ranges, last layers first; ddn_resnet34_8s_grad_buckets lists them).
 * ------------------------------------------------------------------------------------------ */
enum { DDN_MODE_INFER = 0, DDN_MODE_TRAIN = 1, DDN_MODE_EVAL_SAVE = 2 };

size_t ddn_resnet34_8s_workspace_bytes(int B, int H, int W, int D, int mode, int precision);

int ddn_resnet34_8s_forward(const float* x, const float* params, float* buffers, float* y,
                            void* workspace, size_t workspace_bytes,
                            int B, int H, int W, int D,
                            int mode, int bn_groups, float momentum, float eps, int precision,
                            float* low_nhwc_out /* optional [B, H/8*W/8, D]: the low-resolution descriptor map y is upsampled from */,
                            void* stream);

typedef void (*ddn_grad_bucket_fn)(void* user, int bucket, int64_t offset, int64_t numel);

/* dy [B,D,H,W] and / or dlow_nhwc [B, H/8*W/8, D] (the cotangent of low_nhwc_out, produced by the loss kernels that are fused
 * with the upsample): either may be NULL, not both. */
int ddn_resnet34_8s_backward(const float* dy, const float* dlow_nhwc, const float* params, float* grads,
                             void* workspace, size_t workspace_bytes,
                             int B, int H, int W, int D, int mode, int bn_groups, float eps, int precision,
                             ddn_grad_bucket_fn on_bucket, void* user, void* stream);

/* offsets[0..3] = first element of gradient bucket 0..3 (in completion order), offsets[4] = param_count; returns 4.
 * Bucket i covers [offsets[i], offsets[i-1]) for i > 0 and [offsets[0], param_count) for i = 0. */
int ddn_resnet34_8s_grad_buckets(int D, int64_t* offsets, int cap);

/* Optional cache of the tensor-core weight packs (bf16 hi/lo, forward and data-gradient layouts of every conv).
 * The caller owns `cache` (ddn_resnet34_8s_weight_cache_bytes(D) bytes of device memory) and bumps `version` whenever the
 * parameter array changed (optimizer step, load_state_dict); forward/backward calls made with the same `params` pointer and
 * `precision` then pack each conv once per version instead of once per call.  cache == NULL switches it off. */
size_t ddn_resnet34_8s_weight_cache_bytes(int D);
int ddn_resnet34_8s_set_weight_cache(void* cache, size_t bytes, const float* params, uint64_t version, int precision);

/* ------------------------------------------------------------------------------------------
 * Pixelwise contrastive loss.
 * Descriptor images are addressed with explicit strides so the reference's strided view
 *   process_network_output: [N,D,H,W].view(N,D,W*H).permute(0,2,1)
 *   (dense_correspondence_network.py:303-319)
 * is consumed in place: element (image b, pixel p, channel c) = base[b*stride_b + p*stride_p + c*stride_c].
 *
 * A "term" is one list of index pairs scored one way:
 *   kind DDN_TERM_MATCH    sum_i ||A[a_i]-B[b_i]||^2                 pixelwise_contrastive_loss.py:131-167
 *   kind DDN_TERM_HINGE    sum_j max(0, M-||A[a_j]-B[b_j]||)^2       :170-213, :271-304
 *   kind DDN_TERM_HINGE_INV    max(0, ||.||-M)^2   (invert=True)     :204-208
 *   flag DDN_TERM_PIXEL_WEIGHT multiplies l_j by min(||uv(gt_b[j/k]) - uv(b_j)||, M_pixel)/M_pixel,
 *        k = n / n_gt                                                :215-269, :307-352
 * Per (image pair, term) the forward produces the fp64 sum and the number of non-zero hinge
 * values ("hard negatives", :210-211) without any host synchronisation.
 * ------------------------------------------------------------------------------------------ */
enum { DDN_TERM_MATCH = 0, DDN_TERM_HINGE = 1, DDN_TERM_HINGE_INV = 2 };
enum { DDN_TERM_PIXEL_WEIGHT = 1 };

typedef struct {
  const int64_t* idx_a; /* [B, n] flat pixel indices into image A (n = u + W*v)                */
  const int64_t* idx_b; /* [B, n]                                                               */
  const int64_t* gt_b;  /* [B, n_gt] matches_b, only read when DDN_TERM_PIXEL_WEIGHT is set      */
  int64_t n;
  int64_t n_gt;
  int32_t kind;
  int32_t flags;
  float margin;  /* M_descriptor of this term */
  float m_pixel; /* M_pixel                   */
  /* Ragged batches (real SpartanDataset samples have a different number of matches per pair: num_matching_attempts is
   * only an upper bound, dense_correspondence/dataset/spartan_dataset_masked.py:652-660,841-858): rows are padded to n
   * (n_gt) with -1 and len[b] (len_gt[b]) gives pair b's true count.  DEVICE pointers [B], NULL = every pair has n (n_gt). */
  const int64_t* len;
  const int64_t* len_gt;
} ddn_loss_term;

#define DDN_MAX_TERMS 8

/* sums  [B, n_terms] fp64, counts [B, n_terms] int64 (both written, not accumulated). */
int ddn_contrastive_terms_forward(const float* pred_a, const float* pred_b,
                                  int64_t stride_b, int64_t stride_p, int64_t stride_c,
                                  int B, int64_t P, int D, int image_width,
                                  const ddn_loss_term* terms_host, int n_terms,
                                  double* sums, int64_t* counts, void* stream);

/* dpred_a/b += sum_t coef[b,t] * d(term_t sum of pair b)/dpred   (scatter-add; caller zero-fills).
 * coef [B, n_terms] fp32 lives on the device so the scale 1/max(#hard,1) never visits the host. */
int ddn_contrastive_terms_backward(const float* pred_a, const float* pred_b,
                                   int64_t stride_b, int64_t stride_p, int64_t stride_c,
                                   int B, int64_t P, int D, int image_width,
                                   const ddn_loss_term* terms_host, int n_terms,
                                   const float* coef, const float* upstream /* device scalar or NULL */,
                                   float* dpred_a, float* dpred_b, void* stream);

/* The same two entry points FUSED WITH THE BILINEAR UPSAMPLE that produced the descriptor images
 * (nn.functional.upsample_bilinear, resnet_dilated.py:320): low_a / low_b [B, h*w, D] are the low-resolution maps
 * (`low_nhwc_out` of ddn_resnet34_8s_forward), index tensors still address the H x W image.  Each descriptor is blended from
 * its 4 low-resolution cells (identical fp32 arithmetic to ddn_upsample_bilinear_forward), so sums / counts equal those of
 * the entry points above on the upsampled image; the backward scatters into d(low) [B, h*w, D] (caller zero-fills), which
 * ddn_resnet34_8s_backward takes as `dlow_nhwc` -- the full-resolution image and its gradient are never touched. */
int ddn_contrastive_terms_forward_lowres(const float* low_a, const float* low_b, int B, int h, int w, int H, int W, int D,
                                         const ddn_loss_term* terms_host, int n_terms,
                                         double* sums, int64_t* counts, void* stream);
int ddn_contrastive_terms_backward_lowres(const float* low_a, const float* low_b, int B, int h, int w, int H, int W, int D,
                                          const ddn_loss_term* terms_host, int n_terms,
                                          const float* coef, const float* upstream,
                                          float* dlow_a, float* dlow_b, void* stream);

/* loss_composer.get_within_scene_loss (dense_correspondence/loss_functions/loss_composer.py:70-143)
 * evaluated on the device from the sums/counts of terms ordered {match, masked, background[, blind]}:
 *   five [5] fp32 = (loss, match_loss, masked_scaled, background_scaled, blind_scaled), mean over B pairs
 *   coef [B, n_terms] fp32 = d(loss)/d(term sum) for the backward above (already divided by B, times upstream). */
typedef struct {
  float match_loss_weight;
  float non_match_loss_weight;
  int32_t scale_by_hard_negatives;
  int32_t has_blind;
  int64_t n_match, n_masked, n_background, n_blind;
  /* ragged batches: per-pair true counts, DEVICE pointers [B] (NULL = the n_* above for every pair) */
  const int64_t* len_match; const int64_t* len_masked; const int64_t* len_background; const int64_t* len_blind;
} ddn_within_scene_cfg;

int ddn_within_scene_compose(const double* sums, const int64_t* counts, int B, int n_terms,
                             const ddn_within_scene_cfg* cfg_host, float* five, float* coef, void* stream);

/* ------------------------------------------------------------------------------------------
 * Host-buffer entry point (pageable or pinned host memory in, host memory out); it stages through
 * device memory it allocates itself and synchronises before returning.
 * ddn_within_scene_loss_host == loss_composer.get_loss(...) for SINGLE_OBJECT_WITHIN_SCENE on
 * descriptor images held on the host; used by the C smoke test and INTEGRATION.md's ctypes stub.
 * ------------------------------------------------------------------------------------------ */
int ddn_within_scene_loss_host(const float* pred_a_host, const float* pred_b_host, /* [B,D,H*W] NCHW */
                               int B, int H, int W, int D,
                               const int64_t* matches_a_host, const int64_t* matches_b_host, int64_t n_match,
                               const int64_t* masked_a_host, const int64_t* masked_b_host, int64_t n_masked,
                               const int64_t* background_a_host, const int64_t* background_b_host, int64_t n_background,
                               float m_masked, float m_background,
                               float match_loss_weight, float non_match_loss_weight, int scale_by_hard_negatives,
                               float* five_host /* [5] */);

/* ------------------------------------------------------------------------------------------
 * Single-operator entry points (unit tests, and the building blocks the two network calls use).
 * Activations are NHWC fp32 inside the library; conv weights arrive in the reference's
 * [Cout, Cin, kh, kw] layout and are repacked on the device.
 * ------------------------------------------------------------------------------------------ */
/* y[N,Ho,Wo,Cout] = conv2d(x[N,H,W,Cin], w[Cout,Cin,k,k], stride, pad, dilation), no bias -- nn.Conv2d (resnet.py:36,136,210) */
int ddn_conv2d_forward(const float* x_nhwc, const float* w_oihw, float* y_nhwc,
                       int N, int H, int W, int Cin, int Cout, int k, int stride, int pad, int dil,
                       int precision, void* workspace, size_t workspace_bytes, void* stream);
size_t ddn_conv2d_workspace_bytes(int N, int H, int W, int Cin, int Cout, int k, int stride, int pad, int dil, int precision);
/* dx (may be NULL) and dw[Cout,Cin,k,k] (overwritten) for the cotangent dy[N,Ho,Wo,Cout]. */
int ddn_conv2d_backward(const float* x_nhwc, const float* w_oihw, const float* dy_nhwc,
                        float* dx_nhwc, float* dw_oihw,
                        int N, int H, int W, int Cin, int Cout, int k, int stride, int pad, int dil,
                        int precision, void* workspace, size_t workspace_bytes, void* stream);

/* Training-mode BatchNorm2d + optional residual + optional ReLU on NHWC (resnet.py:57-67):
 *   y = relu?( (x-mean)/sqrt(var+eps)*gamma + beta + residual? ); mean/var of this batch (biased);
 *   save_mean/save_invstd [C] written; running stats updated when running_mean != NULL. */
int ddn_batchnorm_forward(const float* x, const float* gamma, const float* beta, const float* residual,
                          float* y, float* save_mean, float* save_invstd,
                          float* running_mean, float* running_var,
                          int64_t M, int C, int relu, int training, float momentum, float eps,
                          void* workspace, size_t workspace_bytes, void* stream);
/* g = dy * (y>0 if relu); dx, dgamma, dbeta; d_residual (= g, may be NULL). */
int ddn_batchnorm_backward(const float* dy, const float* x, const float* y, const float* gamma,
                           const float* save_mean, const float* save_invstd,
                           float* dx, float* dgamma, float* dbeta, float* d_residual,
                           int64_t M, int C, int relu, void* workspace, size_t workspace_bytes, void* stream);
size_t ddn_batchnorm_workspace_bytes(int64_t M, int C);

/* Bilinear align_corners=True resize of planar maps [N*C, h, w] -> [N*C, H, W]
 * (nn.functional.upsample_bilinear, resnet_dilated.py:320) and its adjoint. */
int ddn_upsample_bilinear_forward(const float* x, float* y, int NC, int h, int w, int H, int W, void* stream);
int ddn_upsample_bilinear_backward(const float* dy, float* dx, int NC, int h, int w, int H, int W, void* stream);

/* Data-parallel helpers on the flat gradient: g *= scale (after an all-reduce SUM over ranks). */
int ddn_scale_inplace(float* g, int64_t n, float scale, void* stream);

/* Batched best-match search: for each of Q query descriptors [Q,D] find the pixel of the descriptor image res_b
 * (element (p, c) at p*stride_p + c*stride_c, p = u + W*v) with the smallest L2 distance -- the device-side equivalent of
 * DenseCorrespondenceNetwork.find_best_match (dense_correspondence/network/dense_correspondence_network.py:488-525), first
 * minimum on ties like numpy.argmin.  best_uv [Q,2] int64 = (u, v), best_diff [Q] = that distance; norm_diffs (optional)
 * [Q, H*W] = the full distance maps.  mask_b (optional, [H*W] fp32, 1 inside / 0 outside the object mask): additionally
 * the best match restricted to the mask, argmin(norm_diffs + (1 - mask_b) * 1e6) like
 * dense_correspondence/evaluation/evaluation.py:1052-1059 -> best_uv_masked [Q,2], best_diff_masked [Q] (the masked
 * minimum itself, +1e6 outside).  scratch: 2 x Q x 8 bytes. */
int ddn_find_best_match(const float* res_b, int64_t stride_p, int64_t stride_c, int H, int W, int D,
                        const float* queries, int Q, int64_t* best_uv, float* best_diff, float* norm_diffs,
                        const float* mask_b, int64_t* best_uv_masked, float* best_diff_masked,
                        void* scratch, void* stream);

/* Non-match sampling on the device: out_b[j] = flat index (u + W*v) of a pixel drawn uniformly from the nonzero pixels of
 * `mask` [H*W] fp32 (nz[floor(rand_u[j] * #nonzero)], nonzero pixels in ascending order) or, when mask is NULL or empty,
 * from the whole image (floor(rand_u*W), floor(rand_v*H)); out_a[j] = matches_a[j / non_matches_per_match] (may be NULL).
 * == create_non_correspondences (dense_correspondence/correspondence_tools/correspondence_finder.py:276-405, whose
 * "too close" perturbation is a no-op upstream) + create_non_matches / flatten_uv_tensor
 * (dense_correspondence/dataset/spartan_dataset_masked.py:841-858,1255-1264), given the same uniform numbers. */
size_t ddn_sample_non_matches_scratch_bytes(int H, int W);
int ddn_sample_non_matches(const float* mask, int H, int W, const float* rand_u, const float* rand_v, int64_t n,
                           const int64_t* matches_a, int64_t non_matches_per_match, int64_t* out_a, int64_t* out_b,
                           void* scratch, size_t scratch_bytes, void* stream);

/* Pinhole reprojection match finder for candidate pixels of image A == batch_find_pixel_correspondences
 * (dense_correspondence/correspondence_tools/correspondence_finder.py:409-619): zero-depth, field-of-view and occlusion
 * (3 mm margin) pruning, survivors in candidate order.  depth_* are fp32 [H*W] device arrays in raw sensor units
 * (millimetres, DEPTH_IM_SCALE = 1000); K [9], pose_a [16], pose_b [16] are row-major HOST doubles (camera-to-world poses).
 * out_a / out_b [n] int64 flat pixels (u + W*v; b truncated like .long()), out_u2 / out_v2 optional sub-pixel positions in B;
 * *out_count (DEVICE int64) = number of survivors. */
size_t ddn_find_pixel_correspondences_scratch_bytes(int64_t n);
int ddn_find_pixel_correspondences(const float* depth_a, const float* depth_b, int H, int W,
                                   const int64_t* candidates, int64_t n,
                                   const double* K_host, const double* pose_a_host, const double* pose_b_host,
                                   int64_t* out_a, int64_t* out_b, float* out_u2, float* out_v2, int64_t* out_count,
                                   void* scratch, size_t scratch_bytes, void* stream);

/* Fused Adam step over flat arrays == torch.optim.Adam(lr, betas, eps, weight_decay) as used by
 * dense_correspondence/training/training.py:133-145,346 (L2 weight decay folded into the gradient, bias-corrected moments,
 * no amsgrad).  `step` is the 1-based step count; grads are read as grads[i]*grad_scale (1/world after a SUM all-reduce). */
int ddn_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, int64_t step,
                  float lr, float beta1, float beta2, float eps, float weight_decay, float grad_scale, void* stream);

/* Per-kernel-class device timing (CUDA events recorded on the launching stream around each launch of the
 * convolution / loss kernels while enabled).  ddn_profile_read synchronises on the recorded events and
 * fills one entry per class that ran: work = algorithmic FLOPs (conv_*) or bytes (loss_*). */
typedef struct {
  char name[32];
  int64_t launches;
  double ms;
  double work;
} ddn_profile_entry;
int ddn_profile_enable(int on);
int ddn_profile_reset(void);
int ddn_profile_read(ddn_profile_entry* out, int cap);

/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
int64_t ddn_kernel_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* DDN_B200_H_ */
